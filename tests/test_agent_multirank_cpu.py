"""The N>1 path of the validated agent on CPU: two `gloo` ranks, each running rl_games_b200.agent.A2CAgent (host logic, torch stand-ins
for the kernels, `b200_fused_allreduce: False` so the exchange is a plain `dist.all_reduce` like on the NCCL fallback path) on its OWN
experience, checked against the oracle restatement driven by the same collectives (a2c_common.py:493-509 flat gradient SUM / world,
:1559-1561 KL mean, :782-808 pooled running-stat merge).  Proves: ranks stay byte-identical, gradients and KL are averaged not summed,
the LR schedule follows the rank-mean KL, the normalisers end up with the pooled moments."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')


class _Patch:
    """monkeypatch.setattr look-alike for the spawned workers (the processes end with the test)"""

    def setattr(self, target, name, value):
        setattr(target, name, value)


def _rank_tapes(g, rank):
    """rank 0 replays the fixture's tapes, rank 1 a different experience of the same shape (envs reversed, time rolled)"""
    if rank == 0:
        return g
    g = dict(g)
    for k in ('obs_tape', 'done_tape', 'timeout_tape'):
        g[k] = torch.roll(torch.flip(g[k], dims=[1]), shifts=3, dims=0).contiguous()
    g['obs_tape'] = g['obs_tape'] * 1.5 + 0.25
    g['noise'] = [torch.flip(n, dims=[1]).contiguous() for n in g['noise']]
    return g


def _init_rank(rank, world, port):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    # multi_gpu: True makes the agent name its device 'cuda:<local_rank>' (a2c_common.py:206-220): map that to the CPU in this process
    real_device = torch.device

    class _Meta(type):
        def __instancecheck__(cls, obj):
            return isinstance(obj, real_device)

    class _Dev(metaclass=_Meta):
        def __new__(cls, *a, **k):
            if a and isinstance(a[0], str) and a[0].startswith('cuda'):
                return real_device('cpu')
            return real_device(*a, **k)

    torch.device = _Dev


def _worker(rank, world, port, ret, runs, name='agent_masked.pt', extra=None):
    _init_rank(rank, world, port)
    import test_agent_host_cpu as H
    from oracle import ppo_oracle as O
    from test_oracle_vs_golden import _oracle_from_golden
    g = _rank_tapes(torch.load(os.path.join(GOLDEN, name), weights_only=False), rank)
    agent = H._build(_Patch(), os.path.join(runs, str(rank)), g, H._Env(g),
                     over={'multi_gpu': True, 'b200_fused_allreduce': False, 'print_stats': False, **(extra or {})})
    assert agent.multi_gpu and agent.world_size == 2 and agent.global_rank == rank and not agent.fused_allreduce
    ar = lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM)      # noqa: E731
    orc = _oracle_from_golden(g)
    orc.all_reduce, orc.world_size = ar, world
    snaps = {}
    out = []
    for ep in range(len(g['epochs_out'])):
        agent.epoch_num += 1
        agent.train_epoch(noise=g['noise'][ep])
        o = orc.train_epoch(g['noise'][ep])
        for name, m in (('obs', orc.model.running_mean_std), ('val', orc.model.value_mean_std)):      # sync_running_stats, pooled mode
            snaps[name] = O.merge_rank_stats(m, ar, snaps.get(name))
        sd = agent.model.state_dict()
        for k in O.param_names(len(g['units']), separate=bool((g.get('network_over') or {}).get('separate', False))):
            torch.testing.assert_close(sd[k], orc.model.p[k].detach(), rtol=1e-3, atol=2e-5, msg=lambda m: f'rank {rank} epoch {ep} {k}: {m}')
        if agent.model.grad_mask is not None:          # separate trunks: the structural zeros survive the averaged update on every rank
            assert float(agent.model.flat[agent.model.grad_mask == 0].abs().max()) == 0.0
        assert agent.last_lr == pytest.approx(orc.last_lr, rel=1e-12)
        torch.testing.assert_close(agent.last_stats[:, 4], torch.stack(o['kl']), rtol=2e-3, atol=1e-7)       # per-rank KL (before the mean)
        for pre, m in (('running_mean_std.', orc.model.running_mean_std), ('value_mean_std.', orc.model.value_mean_std)):
            assert int(sd[pre + 'count']) == int(m.count)
            torch.testing.assert_close(sd[pre + 'running_mean'], m.running_mean.reshape(-1), rtol=1e-6, atol=1e-7)
            torch.testing.assert_close(sd[pre + 'running_var'], m.running_var.reshape(-1), rtol=1e-5, atol=1e-7)
        out.append((agent.model.flat.clone(), agent.last_lr, int(sd['running_mean_std.count']), sd['running_mean_std.running_mean'].clone(),
                    agent.rewards.clone()))
    ret[rank] = out
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('name,extra', [('agent_masked.pt', None),
                                        ('agent_sched_standard.pt', {}),        # one scheduler step per mini-epoch on the rank-mean of the mean KL
                                        ('agent_minsigma.pt', None),            # sigma floor: the chained log-std gradient is what gets averaged
                                        ('agent_separate.pt', None)],           # separate trunks: the masked gradient is what gets averaged
                         ids=['per-minibatch schedule', 'per-mini-epoch schedule', 'min_sigma', 'separate trunks'])
def test_two_rank_agent_matches_oracle_and_ranks_stay_identical(name, extra, tmp_path):
    world, port = 2, 29500 + (os.getpid() + len(name)) % 400
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, ret, str(tmp_path), name, extra), nprocs=world, join=True)
    g = torch.load(os.path.join(GOLDEN, name), weights_only=False)
    for ep in range(len(g['epochs_out'])):
        (p0, lr0, c0, m0, r0), (p1, lr1, c1, m1, r1) = ret[0][ep], ret[1][ep]
        assert torch.equal(p0, p1) and lr0 == lr1                      # same averaged gradient, same schedule -> byte-identical weights
        assert c0 == c1 and torch.equal(m0, m1)                       # pooled normaliser state
        assert not torch.equal(r0, r1)                                # ... from different experience
    # two ranks on different data: not the single-rank golden run any more (flat arena = sigma[A] then actor_mlp.0.weight, ...)
    w0 = g['epochs_out'][-1]['state']['a2c_network.actor_mlp.0.weight'].reshape(-1)
    off = (g['A'] + 7) // 8 * 8                                       # arena tensors start on 8-element boundaries (model.py)
    assert not torch.allclose(ret[0][-1][0][off:off + w0.numel()], w0, rtol=1e-3, atol=1e-5)


def _worker_cv(rank, world, port, ret, runs):
    """central value (gated path): the critic has its OWN per-minibatch gradient exchange (central_value.py:322-337) and its normalisers
    join the pooled stats sync (a2c_common.py:753-765)"""
    _init_rank(rank, world, port)
    import test_agent_cv_host_cpu as HC
    from oracle import ppo_oracle as O
    from test_oracle_vs_golden import _cv_oracle_from_golden
    g = _rank_tapes(torch.load(os.path.join(GOLDEN, 'agent_cv.pt'), weights_only=False), rank)
    if rank:
        g['state_tape'] = torch.roll(torch.flip(g['state_tape'], dims=[1]), shifts=3, dims=0).contiguous() * 0.75 - 0.1
        g['noise'] = torch.flip(torch.stack(list(g['noise'])), dims=[2]).contiguous()
    agent = HC._build_cv(_Patch(), os.path.join(runs, str(rank)), g,
                         over={'multi_gpu': True, 'b200_fused_allreduce': False, 'print_stats': False})
    cv = agent.central_value_net
    assert agent.multi_gpu and cv.multi_gpu and cv.world_size == 2
    ar = lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM)      # noqa: E731
    orc, ocv = _cv_oracle_from_golden(g)
    orc.all_reduce, orc.world_size = ar, world
    ocv.all_reduce, ocv.world_size = ar, world
    snaps, out = {}, []
    flat_noise = g['noise'].reshape(-1, g['N'], g['A'])
    for ep in range(len(g['epochs_out'])):
        nz = flat_noise[ep * g['H']:(ep + 1) * g['H']]
        agent.epoch_num += 1
        agent.train_epoch(noise=nz)
        orc.train_epoch(nz)
        for name, m in (('obs', orc.model.running_mean_std), ('val', orc.model.value_mean_std), ('cv_obs', ocv.running_mean_std),
                        ('cv_val', ocv.value_mean_std)):
            snaps[name] = O.merge_rank_stats(m, ar, snaps.get(name))
        sd, csd = agent.model.state_dict(), cv.state_dict()
        for k in O.param_names(len(g['units'])):
            torch.testing.assert_close(sd[k], orc.model.p[k].detach(), rtol=1e-3, atol=2e-5, msg=lambda m: f'rank {rank} epoch {ep} {k}: {m}')
        for k in g['cv_param_order']:
            torch.testing.assert_close(csd[k], ocv.p[k].detach(), rtol=1e-3, atol=2e-5, msg=lambda m: f'rank {rank} epoch {ep} cv {k}: {m}')
        assert agent.last_lr == pytest.approx(orc.last_lr, rel=1e-12) and cv.lr == pytest.approx(ocv.lr, rel=1e-12)
        for pre, m in (('running_mean_std.', ocv.running_mean_std), ('value_mean_std.', ocv.value_mean_std)):
            assert int(csd[pre + 'count']) == int(m.count)
            torch.testing.assert_close(csd[pre + 'running_mean'], m.running_mean.reshape(-1), rtol=1e-6, atol=1e-7)
            torch.testing.assert_close(csd[pre + 'running_var'], m.running_var.reshape(-1), rtol=1e-5, atol=1e-7)
        assert int(sd['running_mean_std.count']) == int(orc.model.running_mean_std.count)
        out.append((agent.model.flat.clone(), cv.flat.clone(), csd['running_mean_std.running_mean'].clone(), int(csd['value_mean_std.count'])))
    ret[rank] = out
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_central_value_agent_matches_oracle_and_ranks_stay_identical(tmp_path):
    world, port = 2, 29900 + os.getpid() % 90
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker_cv, args=(world, port, ret, str(tmp_path)), nprocs=world, join=True)
    for (p0, c0, m0, n0), (p1, c1, m1, n1) in zip(ret[0], ret[1]):
        assert torch.equal(p0, p1) and torch.equal(c0, c1) and torch.equal(m0, m1) and n0 == n1


def _worker_discrete(rank, world, port, ret, runs):
    """discrete PPO (gated path): NCCL-style flat-gradient all-reduce in front of the Adam kernel, rank-mean KL for the per-mini-epoch
    scheduler (a2c_common.py:1272-1274), pooled normaliser sync"""
    _init_rank(rank, world, port)
    import test_discrete_host_cpu as HD
    from oracle import ppo_oracle as O
    from test_oracle_vs_golden import _discrete_oracle_from_golden
    g = torch.load(os.path.join(GOLDEN, 'agent_discrete_masked.pt'), weights_only=False)
    if rank:
        g = dict(g)
        for k in ('obs_tape', 'done_tape', 'timeout_tape', 'mask_tape'):
            g[k] = torch.roll(torch.flip(g[k], dims=[1]), shifts=2, dims=0).contiguous()
        g['u'] = torch.flip(g['u'], dims=[-1]).contiguous()
    agent = HD._build(_Patch(), os.path.join(runs, str(rank)), g, over={'multi_gpu': True, 'print_stats': False})
    assert agent.multi_gpu and agent.world_size == 2 and agent.global_rank == rank
    ar = lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM)      # noqa: E731
    orc = _discrete_oracle_from_golden(g)
    orc.all_reduce, orc.world_size = ar, world
    snaps, out = {}, []
    for ep in range(len(g['epochs_out'])):
        agent.epoch_num += 1
        agent.train_epoch(u=g['u'][ep])
        orc.train_epoch(g['u'][ep])
        for name, m in (('obs', orc.model.running_mean_std), ('val', orc.model.value_mean_std)):
            if m is not None:
                snaps[name] = O.merge_rank_stats(m, ar, snaps.get(name))
        sd = agent.model.state_dict()
        for k in g['param_order']:
            torch.testing.assert_close(sd[k], orc.model.p[k].detach(), rtol=1e-3, atol=2e-5, msg=lambda m: f'rank {rank} epoch {ep} {k}: {m}')
        assert agent.last_lr == pytest.approx(orc.last_lr, rel=1e-12)
        if orc.model.running_mean_std is not None:
            assert int(sd['running_mean_std.count']) == int(orc.model.running_mean_std.count)
            torch.testing.assert_close(sd['running_mean_std.running_mean'], orc.model.running_mean_std.running_mean.reshape(-1), rtol=1e-6, atol=1e-7)
        out.append((agent.model.flat.clone(), agent.last_lr, agent.actions.clone()))
    ret[rank] = out
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_discrete_agent_matches_oracle_and_ranks_stay_identical(tmp_path):
    world, port = 2, 30100 + os.getpid() % 90
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker_discrete, args=(world, port, ret, str(tmp_path)), nprocs=world, join=True)
    for (p0, lr0, a0), (p1, lr1, a1) in zip(ret[0], ret[1]):
        assert torch.equal(p0, p1) and lr0 == lr1 and not torch.equal(a0, a1)
