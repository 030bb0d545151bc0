"""Discrete-action PPO on the GPU (SURVEY 8a row a15): kernels rl_games_b200/csrc/discrete.cu, agent rl_games_b200/agent_discrete.py;
first green on a B200 in round 2.  The oracle side (oracle/ppo_discrete_oracle.py) is pinned to the real reference by
tests/test_oracle_vs_golden.py, which runs on CPU."""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import ppo_discrete_oracle as DO

pytestmark = [pytest.mark.gpu]
DEV = 'cuda:0'
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
RUNS = tempfile.TemporaryDirectory(prefix='b200_test_runs_')      # the agents' train_dir: private to this process, removed at exit


@pytest.mark.parametrize('masked,fused', [(False, True), (True, True), (True, False)])
def test_categorical_sample_vs_oracle(masked, fused):
    """rollout head: actions bit-exact except on cdf boundaries (none expected at these sizes), neglogp / values 1e-5"""
    from rl_games_b200 import ops
    g = torch.Generator().manual_seed(3)
    N, K = 1000, 7
    head = torch.randn(N, 1 + K, generator=g) * 2
    masks = None
    if masked:
        masks = torch.rand(N, K, generator=g) < 0.6
        masks[torch.arange(N), torch.randint(0, K, (N,), generator=g)] = True
    u = torch.rand(N, generator=g)
    nl, probs, _ = DO.categorical_masked(head[:, 1:], masks)
    a_ref = DO.sample_inverse_cdf(probs, u)
    nlp_ref = -nl.gather(1, a_ref.unsqueeze(1)).squeeze(1)
    hd = head.to(DEV)
    if fused:
        lg, ld, vl, vld = hd[:, 1:], 1 + K, hd, 1 + K
    else:
        lg, ld, vl, vld = hd[:, 1:].contiguous(), K, hd[:, :1].contiguous(), 1
    actions = torch.zeros(N, dtype=torch.int64, device=DEV); nlp = torch.zeros(N, device=DEV); vals = torch.zeros(N, device=DEV)
    vm, vv = torch.tensor([1.5], dtype=torch.float64, device=DEV), torch.tensor([4.0], dtype=torch.float64, device=DEV)
    ops.categorical_sample(lg, ld, K, vl, vld, None if masks is None else masks.to(torch.uint8).to(DEV), u.to(DEV), 0, None, 0, vm, vv, True,
                           actions, nlp, vals, None, None, None, None, N)
    torch.cuda.synchronize()
    assert (actions.cpu() == a_ref).float().mean() > 0.998
    same = actions.cpu() == a_ref
    torch.testing.assert_close(nlp.cpu()[same], nlp_ref[same], rtol=1e-5, atol=1e-5)
    if masks is not None:
        assert masks.gather(1, actions.cpu().unsqueeze(1)).all()
    v_ref = (4.0 + 1e-5) ** 0.5 * head[:, 0].clamp(-5, 5) + 1.5
    torch.testing.assert_close(vals.cpu(), v_ref, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize('masked', [False, True])
def test_categorical_loss_and_gradients_vs_autograd(masked):
    """training head: per-minibatch loss pieces and d(loss)/d(logits, value) against autograd on the oracle functions"""
    from rl_games_b200 import ops
    from oracle.ppo_oracle import actor_loss, critic_loss, apply_masks
    g = torch.Generator().manual_seed(5)
    M, K = 777, 5
    logits = (torch.randn(M, K, generator=g) * 1.5).requires_grad_(True)
    value = torch.randn(M, 1, generator=g).requires_grad_(True)
    amask = None
    if masked:
        amask = torch.rand(M, K, generator=g) < 0.7
        amask[torch.arange(M), torch.randint(0, K, (M,), generator=g)] = True
    nl, probs, ent = DO.categorical_masked(logits, amask)
    actions = DO.sample_inverse_cdf(probs.detach(), torch.rand(M, generator=g))
    old_nlp = (-nl.detach().gather(1, actions.unsqueeze(1)).squeeze(1) + torch.randn(M, generator=g) * 0.2)
    adv, old_v, ret = torch.randn(M, generator=g), torch.randn(M, 1, generator=g), torch.randn(M, 1, generator=g)
    rmask = (torch.rand(M, generator=g) < 0.8).float() if masked else None
    nlp = -nl.gather(1, actions.unsqueeze(1)).squeeze(1)
    a = actor_loss(old_nlp, nlp, adv, True, 0.2, smooth=False)
    c = critic_loss(old_v, value, 0.2, ret, True)
    losses, _ = apply_masks([a.unsqueeze(1), c, ent.unsqueeze(1)], rmask)
    loss = losses[0] + 0.5 * losses[1] * 1.0 - losses[2] * 0.01
    loss.backward()
    kl = 0.5 * (old_nlp - nlp.detach()) ** 2
    kl = (kl * rmask).sum() / rmask.sum() if rmask is not None else kl.mean()
    d = lambda t: None if t is None else t.to(DEV)   # noqa: E731
    dl, dv = torch.zeros(M, K, device=DEV), torch.zeros(M, 1, device=DEV)
    part = torch.zeros((M + 255) // 256, 8, dtype=torch.float64, device=DEV)
    inv = None if rmask is None else torch.tensor([1.0 / float(rmask.sum())], device=DEV)
    cfg = ops.CatLossCfg(0.2, 1.0, 0.01, 1, 0, 1)
    nb = ops.categorical_loss(d(logits.detach()), K, K, d(value.detach()), 1, d(actions), None if amask is None else d(amask.to(torch.uint8)),
                              d(old_v.squeeze(1)), d(ret.squeeze(1)), d(old_nlp), d(adv), d(rmask), M, 0, M, cfg, inv, dl, K, dv, 1, part)
    torch.cuda.synchronize()
    st = part[:nb, :4].sum(0).cpu().float()
    torch.testing.assert_close(st, torch.stack([losses[0], losses[1], losses[2], kl]).detach().float(), rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(dl.cpu(), logits.grad, rtol=1e-3, atol=1e-7)
    torch.testing.assert_close(dv.cpu(), value.grad, rtol=1e-4, atol=1e-8)


class DiscreteTapeEnvGPU:
    def __init__(self, g):
        self.obs_tape, self.done_tape, self.timeout_tape = g['obs_tape'].to(DEV), g['done_tape'].to(DEV), g['timeout_tape'].to(DEV)
        self.mask_tape = None if g['mask_tape'] is None else g['mask_tape'].to(DEV)
        self.K, self.autoreset, self.i = g['K'], g['autoreset'], 0

    def reset(self):
        self.i = 0
        return self.obs_tape[0].clone()

    def get_action_masks(self):
        return self.mask_tape[self.i % self.mask_tape.shape[0]]

    def step(self, actions):
        j0 = self.i % self.obs_tape.shape[0]
        if isinstance(self.K, (list, tuple)):
            off, rew = 0, 0.0
            for j, k in enumerate(self.K):
                rew = rew + (actions[:, j].long() == self.obs_tape[j0][:, off:off + k].argmax(dim=-1)).float() / len(self.K)
                off += k
        else:
            rew = (actions.long() == self.obs_tape[j0][:, :self.K].argmax(dim=-1)).float()
        self.i += 1
        j = self.i % self.obs_tape.shape[0]
        return self.obs_tape[j].clone(), rew, self.done_tape[j].clone(), {'time_outs': self.timeout_tape[j].clone()}

    def get_env_info(self):
        from rl_games_b200.common import Box, Discrete, Tuple
        space = Tuple([Discrete(k) for k in self.K]) if isinstance(self.K, (list, tuple)) else Discrete(self.K)
        info = {'observation_space': Box(-np.inf, np.inf, (self.obs_tape.shape[-1],)), 'action_space': space}
        if self.autoreset != 'same_step':
            info['autoreset_mode'] = self.autoreset
        return info


@pytest.mark.parametrize('name', ['agent_discrete.pt', 'agent_discrete_masked.pt', 'agent_multidiscrete.pt'])
def test_discrete_agent_matches_reference_golden(name):
    """two train_epoch()s of the reference DiscreteA2CAgent (tests/golden/gen_golden.py discrete) vs rl_games_b200.DiscreteA2CAgent"""
    from rl_games_b200.runner import Runner
    g = torch.load(os.path.join(GOLDEN, name), weights_only=False)
    cfgk = g['config']
    env = DiscreteTapeEnvGPU(g)
    config = {k: v for k, v in cfgk.items() if k not in ('device', 'torch_compile')}
    config.update({'device': DEV, 'env_info': env.get_env_info(), 'vec_env': env, 'reward_shaper': {'scale_value': 0.1},
                   'train_dir': RUNS.name, 'lr_schedule': cfgk.get('lr_schedule', None)})
    multi = isinstance(g['K'], (list, tuple))
    network = {'name': 'actor_critic', 'separate': g['separate'], 'space': {'multi_discrete' if multi else 'discrete': None},
               'mlp': {'units': g['units'], 'activation': 'relu', 'initializer': {'name': 'default'}}}
    r = Runner()
    r.load({'params': {'seed': 1, 'algo': {'name': 'a2c_discrete'}, 'model': {'name': 'multi_discrete_a2c' if multi else 'discrete_a2c'},
                       'network': network, 'config': config}})
    r.params['config']['vec_env'] = env
    agent = r.algo_factory.create(r.algo_name, base_name='parity', params=r.params)
    agent.model.load_state_dict({k: v.to(DEV) for k, v in g['init_state'].items()}, strict=False)
    assert agent.model.param_names() == g['param_order']
    agent.init_tensors()
    agent.obs = agent.env_reset()
    fl = lambda t: t.transpose(0, 1).reshape(-1, *t.shape[2:])    # noqa: E731  [H,N,...] -> flat env*H + t
    for ep, ref in enumerate(g['epochs_out']):
        agent.epoch_num += 1
        res = agent.train_epoch(u=g['u'][ep].to(DEV))
        ds = ref['dataset']
        assert (agent.actions.cpu() == ref['mb_actions']).all()
        torch.testing.assert_close(agent.rewards.cpu().unsqueeze(2), ref['mb_rewards'], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(agent.values.cpu().unsqueeze(2), ref['mb_values'], rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(fl(agent.advs_n).cpu(), ds['advantages'], rtol=2e-4, atol=2e-5)
        torch.testing.assert_close(fl(agent.neglogpacs).cpu(), ds['old_logp_actions'], rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(torch.stack(res[4]).cpu(), ref['a_losses'], rtol=2e-3, atol=2e-6)
        torch.testing.assert_close(torch.stack(res[5]).cpu(), ref['c_losses'], rtol=2e-3, atol=2e-6)
        torch.testing.assert_close(torch.stack(res[6]).cpu(), ref['entropies'], rtol=1e-4, atol=1e-6)
        torch.testing.assert_close(torch.stack(res[7]).cpu(), ref['kls'], rtol=5e-3, atol=1e-8)
        assert agent.last_lr == pytest.approx(ref['last_lr'], rel=1e-12)
        sd = agent.model.state_dict()
        for k in g['param_order']:
            torch.testing.assert_close(sd[k].cpu(), ref['state'][k], rtol=1e-3, atol=2e-5, msg=lambda m: k + ': ' + m)
        assert agent.game_rewards.current_size == ref['game_rewards_size']
        torch.testing.assert_close(agent.game_rewards.mean, ref['game_rewards_mean'].reshape(-1), rtol=1e-4, atol=1e-5)


def test_multi_head_kernels_vs_oracle_and_autograd():
    """multi-discrete: heads [3, 4, 2] concatenated; sample kernel vs the oracle rule, loss kernel vs autograd (the same check runs on the
    host-compiled row functions in tests/test_discrete_rows_cpu.py)"""
    from rl_games_b200 import ops
    from oracle.ppo_oracle import actor_loss, critic_loss
    g = torch.Generator().manual_seed(21)
    sizes, M = [3, 4, 2], 900
    K, nh = sum(sizes), len(sizes)
    logits = (torch.randn(M, K, generator=g) * 1.5).requires_grad_(True)
    value = torch.randn(M, 1, generator=g).requires_grad_(True)
    amask = torch.rand(M, K, generator=g) < 0.6
    off = 0
    for k in sizes:
        amask[torch.arange(M), torch.randint(0, k, (M,), generator=g) + off] = True
        off += k
    heads = [DO.categorical_masked(z, m) for z, m in zip(torch.split(logits, sizes, dim=1), torch.split(amask, sizes, dim=1))]
    u = torch.rand(nh, M, generator=g)
    a_ref = torch.stack([DO.sample_inverse_cdf(h[1].detach(), u[j]) for j, h in enumerate(heads)], dim=-1)
    nlp = sum(-h[0].gather(1, a_ref[:, j:j + 1]).squeeze(1) for j, h in enumerate(heads))
    d = lambda t: t.to(DEV)   # noqa: E731
    actions = torch.zeros(M, nh, dtype=torch.int64, device=DEV); nlp_k = torch.zeros(M, device=DEV); vals = torch.zeros(M, device=DEV)
    ops.categorical_sample(d(logits.detach()), K, K, d(value.detach()), 1, d(amask.to(torch.uint8)), d(u.contiguous()), 0, None, 0, None, None,
                           False, actions, nlp_k, vals, None, None, None, None, M, head_sizes=sizes)
    torch.cuda.synchronize()
    same = (actions.cpu() == a_ref).all(dim=1)
    assert same.float().mean() > 0.998
    torch.testing.assert_close(nlp_k.cpu()[same], nlp.detach()[same], rtol=1e-5, atol=1e-5)
    ent = sum(h[2] for h in heads)
    old_nlp = nlp.detach() + torch.randn(M, generator=g) * 0.2
    adv, old_v, ret = torch.randn(M, generator=g), torch.randn(M, 1, generator=g), torch.randn(M, 1, generator=g)
    a = actor_loss(old_nlp, nlp, adv, True, 0.2, smooth=False)
    c = critic_loss(old_v, value, 0.2, ret, True).squeeze(1)
    la, lc, le = a.mean(), c.mean(), ent.mean()
    (la + 0.5 * 1.5 * lc - 0.02 * le).backward()
    dl, dv = torch.zeros(M, K, device=DEV), torch.zeros(M, 1, device=DEV)
    part = torch.zeros((M + 255) // 256, 8, dtype=torch.float64, device=DEV)
    nb = ops.categorical_loss(d(logits.detach()), K, K, d(value.detach()), 1, d(a_ref.contiguous()), d(amask.to(torch.uint8)), d(old_v.squeeze(1)),
                              d(ret.squeeze(1)), d(old_nlp), d(adv), None, M, 0, M, ops.CatLossCfg(0.2, 1.5, 0.02, 1, 0, 1), None, dl, K, dv, 1, part,
                              head_sizes=sizes)
    torch.cuda.synchronize()
    torch.testing.assert_close(part[:nb, :3].sum(0).cpu().float(), torch.stack([la, lc, le]).detach(), rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(dl.cpu(), logits.grad, rtol=1e-3, atol=1e-7)
    torch.testing.assert_close(dv.cpu(), value.grad, rtol=1e-4, atol=1e-8)
