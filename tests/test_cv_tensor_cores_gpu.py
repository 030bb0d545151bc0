"""The tensor-core critic (central_value_config mixed_precision: True) on a B200: the fused value-head kernels of csrc/critic.cu against
float64 autograd and against the kernels they replace, and the critic on the layer-wise tcgen05 GEMMs against the fp32 critic.
Host logic without a GPU: tests/test_cv_tensor_cores_cpu.py."""
import math
import os
import sys
import tempfile

import pytest
import torch

from oracle import ppo_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_cv_gpu import _Env  # noqa: E402

pytestmark = [pytest.mark.gpu]
DEV = 'cuda:0'
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
RUNS = tempfile.TemporaryDirectory(prefix='b200_test_runs_')      # the agents' train_dir: private to this process, removed at exit
ACT = {1: torch.nn.functional.elu, 2: torch.relu, 3: torch.tanh}


def _act_grad(a, act):
    return {1: torch.where(a > 0, torch.ones_like(a), a + 1.0), 2: (a > 0).to(a.dtype), 3: 1.0 - a * a}[act]


def _fill_ff(*ts):
    for t in ts:
        t.view(torch.uint8).fill_(0xFF)          # NaN in every float lane


# (Hl, activation, clip_value, mask, H, N, envs per minibatch, first env, n_splits).  M = H * epm rows in chunks of epm: 128- and
# 256-row blocks straddle the chunks, M is not a multiple of 128; H = 24 gives clusters of several CTAs per split; 16 splits on 305 rows
# leave most splits empty.
HEAD_CASES = [
    (1, 1, True, 'none', 5, 150, 61, 37, 3),
    (7, 2, False, 'random', 5, 150, 61, 37, 3),
    (64, 3, True, 'random', 24, 256, 200, 40, 2),
    (128, 1, False, 'none', 24, 256, 200, 40, 2),
    (512, 2, True, 'zero', 5, 150, 61, 37, 16),
    (1000, 3, False, 'random', 5, 150, 61, 37, 1),
    (128, 1, True, 'random', 24, 256, 200, 40, 16),
    (1000, 1, True, 'none', 24, 256, 200, 40, 2),
]


def _run_head(a, W, b, ov, rt, mk, inv, epm, N, M, clip, act, n_splits, fill_ff):
    from rl_games_b200 import ops
    Hl = W.numel()
    P, off_w = Hl + 1 + 40, 17
    off_b = off_w + Hl
    part = torch.full((n_splits, P), 7.0, device=DEV)
    d_alast = torch.full((M + 3, Hl), 7.0, device=DEV)
    partials = torch.full(((M + 255) // 256 + 2, 8), 7.0, dtype=torch.float64, device=DEV)
    vo = torch.full((M + 1,), 7.0, device=DEV)
    if fill_ff:
        _fill_ff(d_alast[:M], part[:, off_w:off_b + 1], partials[:(M + 255) // 256], vo[:M])
    nb = ops.value_head_loss(a, W, b, ov, rt, mk, epm, N, M, 0.2, clip, inv, act, d_alast, part[0, off_w:], part[0, off_b:], P, n_splits,
                             partials, value_out=vo)
    torch.cuda.synchronize()
    return nb, dict(part=part, d_alast=d_alast, partials=partials, vo=vo, P=P, off_w=off_w, off_b=off_b)


@pytest.mark.parametrize('case', HEAD_CASES, ids=lambda c: 'Hl%d-act%d-clip%d-%s-M%d-S%d' % (c[0], c[1], c[2], c[3], c[4] * c[6], c[8]))
def test_value_head_loss_kernel_vs_float64_autograd(case):
    from rl_games_b200 import ops
    Hl, act, clip, mkind, H, N, epm, e0, S = case
    M = H * epm
    g = torch.Generator().manual_seed(Hl * 7 + act)
    a = ACT[act](torch.randn(M, Hl, generator=g))
    W, b = torch.randn(Hl, generator=g) / math.sqrt(Hl), torch.randn(1, generator=g) * 0.1
    old_v, ret = torch.randn(H, N, generator=g), torch.randn(H, N, generator=g)
    mask = None if mkind == 'none' else ((torch.rand(H, N, generator=g) < 0.7).float() if mkind == 'random' else torch.zeros(H, N))
    sl = lambda t: torch.cat([t[h, e0:e0 + epm] for h in range(H)])   # noqa: E731  minibatch rows in kernel order (chunk-major)
    # float64 reference
    a64, W64 = a.double(), W.double()
    v = (a64 @ W64 + b.double()).requires_grad_(True)
    c = O.critic_loss(sl(old_v).double().unsqueeze(1), v.unsqueeze(1), 0.2, sl(ret).double().unsqueeze(1), clip).squeeze(1)
    inv = None if mask is None else 1.0 / max(float(sl(mask).sum()), 1.0)
    w = torch.full((M,), 1.0 / M, dtype=torch.float64) if mask is None else sl(mask).double() * inv
    loss = (c * w).sum()
    loss.backward()
    dv = v.grad
    d_alast_ref = dv[:, None] * W64[None, :] * _act_grad(a64, act)
    dW_ref, db_ref = (dv[:, None] * a64).sum(0), dv.sum()
    # the kernel
    d = lambda t: None if t is None else t.to(DEV)   # noqa: E731
    ad, Wd, bd, ov, rt, mk = d(a), d(W), d(b), d(old_v), d(ret), d(mask)
    invd = None if mask is None else torch.tensor([inv], device=DEV)
    args = (ad, Wd, bd, ov[0, e0:], rt[0, e0:], None if mk is None else mk[0, e0:], invd, epm, N, M, clip, act, S)
    nb, o = _run_head(*args, fill_ff=False)
    assert nb == (M + 255) // 256
    P, off_w, off_b = o['P'], o['off_w'], o['off_b']
    torch.testing.assert_close(o['d_alast'][:M].cpu().double(), d_alast_ref, rtol=1e-3, atol=1e-5 * float(d_alast_ref.abs().max()) + 1e-12)
    grad = torch.zeros(P, device=DEV)
    ops.reduce_splits(o['part'], grad, P, S)
    torch.cuda.synchronize()
    torch.testing.assert_close(grad[off_w:off_b].cpu().double(), dW_ref, rtol=1e-3, atol=1e-5 * float(dW_ref.abs().max()) + 1e-12)
    assert float(grad[off_b]) == pytest.approx(float(db_ref), rel=1e-3, abs=1e-6)
    pr = o['partials'][:nb].cpu()
    assert float(pr[:, 0].sum()) == pytest.approx(float(loss), rel=1e-5, abs=1e-9)
    assert float(pr[:, 1].sum()) == (M if mask is None else float(sl(mask).sum()))
    assert float(pr[:, 2].sum()) == pytest.approx(float(w.sum()), rel=1e-5, abs=1e-9)
    assert torch.all(pr[:, 3:] == 0)
    torch.testing.assert_close(o['vo'][:M].cpu().double(), v.detach(), rtol=1e-5, atol=1e-5)
    # untouched: arena entries outside the head's slots, rows past M, partial rows past nb, value_out past M
    keep = torch.ones(P, dtype=torch.bool)
    keep[off_w:off_b + 1] = False
    assert torch.all(o['part'][:, keep] == 7.0)
    assert torch.all(o['d_alast'][M:] == 7.0) and torch.all(o['partials'][nb:] == 7.0) and float(o['vo'][M]) == 7.0
    # deterministic, and blind to what the outputs held before: a second run over 0xFF-filled buffers gives the same bytes
    nb2, o2 = _run_head(*args, fill_ff=True)
    assert nb2 == nb
    assert torch.equal(o2['d_alast'][:M], o['d_alast'][:M]) and torch.equal(o2['vo'][:M], o['vo'][:M])
    assert torch.equal(o2['part'][:, off_w:off_b + 1], o['part'][:, off_w:off_b + 1]) and torch.equal(o2['partials'][:nb], o['partials'][:nb])
    # the loss rows are value_loss_f32's, given the same values
    dvv = torch.zeros(M, 1, device=DEV)
    part_vl = torch.zeros(nb, 8, dtype=torch.float64, device=DEV)
    nb3 = ops.value_loss(o['vo'], 1, ov[0, e0:], rt[0, e0:], None if mk is None else mk[0, e0:], epm, N, M, 0.2, clip, invd, dvv, 1, part_vl)
    torch.cuda.synchronize()
    assert nb3 == nb and torch.equal(part_vl, o['partials'][:nb])


@pytest.mark.parametrize('Hl', [1, 7, 128, 1000])
@pytest.mark.parametrize('normalize', [False, True])
def test_value_head_rollout_kernel_vs_linear_fwd_and_normalize(Hl, normalize):
    """one launch = linear_fwd (Nout = 1) + normalize(denorm); the dot product is the training kernel's, bit for bit"""
    from rl_games_b200 import ops
    N = 1000
    g = torch.Generator().manual_seed(Hl)
    a = torch.nn.functional.elu(torch.randn(N, Hl, generator=g)).to(DEV)
    W, b = (torch.randn(Hl, generator=g) / math.sqrt(Hl)).to(DEV), (torch.randn(1, generator=g) * 0.1).to(DEV)
    mean = torch.tensor([0.7], dtype=torch.float64, device=DEV)
    var = torch.tensor([2.3], dtype=torch.float64, device=DEV)
    Y = torch.zeros(N, 1, device=DEV)
    ops.linear_fwd(a, W.view(1, Hl), b, Y, 0, M=N)
    ref = ops.normalize(Y, mean, var, denorm=True).view(-1) if normalize else Y.view(-1)
    got = torch.full((N,), float('nan'), device=DEV)
    ops.value_head_fwd(a, W, b, mean if normalize else None, var if normalize else None, normalize, got, N)
    torch.cuda.synchronize()
    scale = float((a.abs() @ W.abs()).max()) * (math.sqrt(2.3 + 1e-5) if normalize else 1.0)
    torch.testing.assert_close(got, ref, rtol=1e-6, atol=1e-6 * scale)
    # the training kernel's value for the same rows
    z = torch.zeros(N, device=DEV)
    vo = torch.zeros(N, device=DEV)
    ops.value_head_loss(a, W, b, z, z, None, N, 0, N, 0.2, False, None, 1, torch.empty(N, Hl, device=DEV), torch.empty(Hl, device=DEV),
                        torch.empty(1, device=DEV), Hl, 1, torch.empty((N + 255) // 256, 8, dtype=torch.float64, device=DEV), value_out=vo)
    raw = torch.empty(N, device=DEV)
    ops.value_head_fwd(a, W, b, None, None, False, raw, N)
    torch.cuda.synchronize()
    assert torch.equal(raw, vo)


# ---------------------------------------------------------------------------------------------- the agent
def _tapes(N, H, D, S, A, seed):
    g = torch.Generator().manual_seed(seed)
    obs_tape, done_tape, tout_tape = O.make_tapes(H + 1, N, D, seed=seed, p_done=0.05)
    return {'N': N, 'H': H, 'D': D, 'S': S, 'A': A, 'autoreset': 'same_step', 'obs_tape': obs_tape,
            'state_tape': torch.randn(H + 1, N, S, generator=g), 'done_tape': done_tape, 'timeout_tape': tout_tape}


def _cv_agent(g, config, cv_config, units, cv_units, actor_state=None, cv_state=None):
    from rl_games_b200.runner import Runner
    env = _Env(g)
    cv_cfg = dict(cv_config)
    cv_cfg['network'] = {'name': 'actor_critic', 'central_value': True,
                         'mlp': {'units': list(cv_units), 'activation': 'elu', 'initializer': {'name': 'default'}}}
    config = dict(config)
    config.update({'device': DEV, 'env_info': env.get_env_info(), 'vec_env': env, 'reward_shaper': {'scale_value': 1.0},
                   'b200_cuda_graph': False, 'train_dir': RUNS.name, 'central_value_config': cv_cfg})
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': list(units), 'activation': 'elu', 'initializer': {'name': 'default'}}}
    r = Runner()
    r.load({'params': {'seed': 7, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'}, 'network': network,
                       'config': config}})
    r.params['config']['vec_env'] = env
    agent = r.algo_factory.create(r.algo_name, base_name='cvtc', params=r.params)
    if actor_state is not None:
        agent.model.load_state_dict({k: v.to(DEV) for k, v in actor_state.items()}, strict=False)
    if cv_state is not None:
        agent.central_value_net.load_state_dict({k: v.to(DEV) for k, v in cv_state.items()})
    agent.init_tensors()
    agent._repack()
    agent.obs = agent.env_reset()
    return agent


def _compare(f, t, cv_w0):
    """the bf16 tolerance class of test_layerwise_tensor_core_path_tracks_fp32_agent"""
    cf, ct = f.central_value_net, t.central_value_net
    assert not cf.gemm_tc and ct.gemm_tc
    torch.testing.assert_close(t.values, f.values, rtol=0, atol=6e-2)
    lf, lt = torch.stack(cf.last_losses).cpu(), torch.stack(ct.last_losses).cpu()
    torch.testing.assert_close(lt, lf, rtol=0.1, atol=2e-2)
    sdf, sdt = cf.state_dict(), ct.state_dict()
    for k in cf.param_names():
        if k.endswith('weight'):
            du_f = (sdf[k] - cv_w0[k]).flatten().cpu()
            du_t = (sdt[k] - cv_w0[k]).flatten().cpu()
            cos = float(du_f @ du_t / (du_f.norm() * du_t.norm() + 1e-20))
            assert cos > 0.8, (k, cos)


@pytest.mark.parametrize('actor_mp', [False, True], ids=['actor-fp32', 'actor-tc'])
def test_tensor_core_critic_tracks_fp32_critic_on_the_golden_geometry(actor_mp):
    g = torch.load(os.path.join(GOLDEN, 'agent_cv.pt'), weights_only=False)
    cfg = {k: v for k, v in g['config'].items() if k not in ('device', 'torch_compile', 'train_dir')}
    cfg['mixed_precision'] = actor_mp
    flat_noise = g['noise'].reshape(-1, g['N'], g['A']).to(DEV)
    agents = []
    for mp in (False, True):
        a = _cv_agent(g, cfg, dict(g['cv_config'], mixed_precision=mp), g['units'], g['cv_units'], g['init_state'], g['cv_init_state'])
        a.epoch_num += 1
        a.train_epoch(noise=flat_noise[:g['H']])
        agents.append(a)
    _compare(*agents, {k: v.to(DEV) for k, v in g['cv_init_state'].items()})


@pytest.mark.parametrize('actor_mp', [False, True], ids=['actor-fp32', 'actor-tc'])
def test_tensor_core_critic_512_256_128_tracks_fp32_critic(actor_mp):
    """an mjlab-sized critic ([512, 256, 128], minibatch 4096, two minibatches) behind an actor on the fp32 kernels or the fused tcgen05
    kernels ([256, 128, 64], 32 observations)"""
    N, H, D, S, A = 1024, 8, 32, 48, 6
    g = _tapes(N, H, D, S, A, seed=21)
    cfg = {'name': 'cvtc', 'env_name': 'unused', 'multi_gpu': False, 'mixed_precision': actor_mp, 'normalize_input': True,
           'normalize_value': True, 'value_bootstrap': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95, 'learning_rate': 3e-4,
           'lr_schedule': 'adaptive', 'kl_threshold': 0.008, 'grad_norm': 1.0, 'entropy_coef': 0.0, 'truncate_grads': True, 'e_clip': 0.2,
           'clip_value': False, 'max_epochs': 100, 'num_actors': N, 'horizon_length': H, 'minibatch_size': 4096, 'mini_epochs': 2,
           'critic_coef': 1, 'save_frequency': 0, 'print_stats': False}
    cv_cfg = {'minibatch_size': 4096, 'mini_epochs': 3, 'learning_rate': 5e-4, 'clip_value': True, 'normalize_input': True,
              'truncate_grads': True, 'grad_norm': 1.0}
    noise = torch.randn(H, N, A, generator=torch.Generator().manual_seed(5)).to(DEV)
    agents, w0 = [], None
    for mp in (False, True):
        a = _cv_agent(g, cfg, dict(cv_cfg, mixed_precision=mp), [256, 128, 64], [512, 256, 128],
                      actor_state=None if not agents else agents[0]._init_actor, cv_state=w0)
        if not agents:
            a._init_actor = {k: v.clone() for k, v in a.model.state_dict().items()}
            w0 = {k: v.clone() for k, v in a.central_value_net.state_dict().items()}
        assert a.use_tc == actor_mp and a.central_value_net.gemm_tc == mp and a.central_value_net.n_splits == (8 if mp else 16)
        a.epoch_num += 1
        a.train_epoch(noise=noise)
        agents.append(a)
    _compare(*agents, w0)


def test_get_value_follows_a_loaded_checkpoint():
    """the bf16 twin after a load: get_value of a fresh tensor-core critic, restored from another one's checkpoint, equals the trained
    critic's get_value bit for bit (same weights, same twin, same kernels), and not the fresh critic's"""
    N, H, D, S, A = 256, 8, 16, 40, 4
    g = _tapes(N, H, D, S, A, seed=33)
    cfg = {'name': 'cvtc', 'env_name': 'unused', 'multi_gpu': False, 'mixed_precision': False, 'normalize_input': True,
           'normalize_value': True, 'value_bootstrap': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95, 'learning_rate': 3e-4,
           'lr_schedule': None, 'grad_norm': 1.0, 'entropy_coef': 0.0, 'truncate_grads': True, 'e_clip': 0.2, 'clip_value': False,
           'max_epochs': 100, 'num_actors': N, 'horizon_length': H, 'minibatch_size': 1024, 'mini_epochs': 1, 'critic_coef': 1,
           'save_frequency': 0, 'print_stats': False}
    cv_cfg = {'minibatch_size': 1024, 'mini_epochs': 4, 'learning_rate': 3e-3, 'clip_value': False, 'normalize_input': True,
              'mixed_precision': True}
    a = _cv_agent(g, cfg, cv_cfg, [32, 16], [512, 256, 128])
    a.epoch_num += 1
    a.train_epoch()
    path = os.path.join(RUNS.name, 'cvtc_ck')
    a.save(path)
    b = _cv_agent(g, cfg, cv_cfg, [32, 16], [512, 256, 128])
    states = g['state_tape'][0].to(DEV)
    fresh, got, want = (torch.zeros(N, device=DEV) for _ in range(3))
    b.central_value_net.get_value(states, fresh)
    b.restore_central_value_function(path + '.pth')
    b.central_value_net.get_value(states, got)
    a.central_value_net.get_value(states, want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert not torch.allclose(got, fresh, rtol=1e-3, atol=1e-3)
