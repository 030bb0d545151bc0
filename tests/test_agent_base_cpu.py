"""What the continuous and the discrete agents share through rl_games_b200.agent_base.A2CBase, on CPU with torch stand-ins for the
kernels: the rank-0 control flow of train() on two gloo ranks, normaliser history on resume under the pooled cross-rank sync, stop_fn,
env_state in checkpoints and the PBT experiment name."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')


def _golden(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


class _Scalars:
    def __init__(self):
        self.seen = []

    def add_scalar(self, tag, v, step=None):
        self.seen.append(tag)


def _train_worker(rank, world, port, ret, runs, kind):
    """train() to max_epochs 2 on rank `rank` of a two-rank gloo group; returns what train() returned, the checkpoint files and the
    summary tags this rank wrote"""
    from test_agent_multirank_cpu import _Patch, _init_rank
    _init_rank(rank, world, port)
    # the fixtures' save_best_after is out of reach: only rank 0 tracks the best reward, so with a best-reward save the ranks would return
    # different last_mean_rewards (as the reference's do)
    over = {'multi_gpu': True, 'print_stats': False, 'max_epochs': 2, 'save_frequency': 1, 'name': 'two_ranks'}
    if kind == 'continuous':
        import _torch_ops
        import test_agent_host_cpu as H
        from rl_games_b200 import ops
        g = _golden('agent_masked.pt')
        agent = H._build(_Patch(), os.path.join(runs, str(rank)), g, H._Env(g), over={**over, 'b200_fused_allreduce': False})
        tape, orig = g['noise'][0], _torch_ops.policy_head_sample

        def sample_with_tape(*args, **kw):          # train() passes no noise tape: feed one so that the stand-in needs no RNG
            args = list(args)
            if args[7] is None:
                args[7] = tape[int(args[10]) % tape.shape[0]]
            return orig(*args, **kw)
        ops.policy_head_sample = sample_with_tape
    else:
        import test_discrete_host_cpu as HD
        agent = HD._build(_Patch(), os.path.join(runs, str(rank)), _golden('agent_discrete_masked.pt'), over=over)
    assert agent.world_size == 2 and agent.global_rank == rank
    scalars = None
    if agent.writer is not None:
        scalars = _Scalars()
        agent.writer = agent.algo_observer.writer = scalars
    last, epochs = agent.train()
    ret[rank] = (float(last), epochs, sorted(os.listdir(agent.nn_dir)), None if scalars is None else scalars.seen)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('kind', ['continuous', 'discrete'])
def test_two_rank_train_loop_logs_and_checkpoints_on_rank_0_only(kind, tmp_path):
    world, port = 2, 30300 + (os.getpid() + 7 * len(kind)) % 90
    ret = mp.Manager().dict()
    mp.spawn(_train_worker, args=(world, port, ret, str(tmp_path), kind), nprocs=world, join=True)
    (last0, ep0, files0, tags0), (last1, ep1, files1, tags1) = ret[0], ret[1]
    assert ep0 == ep1 == 2 and last0 == last1
    assert any(f.endswith('.pth') for f in files0) and files1 == []
    assert 'losses/a_loss' in tags0 and 'info/epochs' in tags0 and tags1 is None


def _discrete(monkeypatch, tmp_path, over=None, name='agent_discrete_masked.pt'):
    import test_discrete_host_cpu as HD
    return HD._build(monkeypatch, tmp_path, _golden(name), over=over)


def test_discrete_resume_under_pooled_sync_counts_the_restored_history_once(monkeypatch, tmp_path):
    """two identical ranks, stood in for by an all-reduce that doubles its tensor: after a restore, the first pooled merge adds each
    rank's NEW rows only (a2c_common.py:767-780), not the restored history once per rank"""
    g = _golden('agent_discrete_masked.pt')
    a = _discrete(monkeypatch, tmp_path / 'a')
    a.epoch_num += 1
    a.train_epoch(u=g['u'][0])
    fn = str(tmp_path / 'ck')
    a.save(fn)
    counts = lambda ag: (int(ag.model.running_mean_std.count), int(ag.model.value_mean_std.count))     # noqa: E731
    restored = counts(a)
    single = _discrete(monkeypatch, tmp_path / 'b')
    single.restore(fn + '.pth')
    single.train_epoch(u=g['u'][1])
    added = [s - c for s, c in zip(counts(single), restored)]
    assert all(n > 0 for n in added)
    two = _discrete(monkeypatch, tmp_path / 'c')
    two.multi_gpu, two.world_size = True, 2
    monkeypatch.setattr(dist, 'all_reduce', lambda t, op=None: t.mul_(2))
    two.restore(fn + '.pth')
    assert counts(two) == restored
    two.train_epoch(u=g['u'][1])
    assert list(counts(two)) == [c + 2 * n for c, n in zip(restored, added)]


def test_discrete_stop_fn_is_an_attribute_checked_at_construction(monkeypatch, tmp_path):
    with pytest.raises(ValueError, match='stop_fn'):
        _discrete(monkeypatch, tmp_path, over={'stop_fn': 'not callable'})
    agent = _discrete(monkeypatch, tmp_path, over={'max_epochs': 5, 'print_stats': False, 'name': 'stopped'})
    agent.stop_fn = lambda ag: ag.epoch_num >= 1
    last, epochs = agent.train()
    assert epochs == 1 and os.listdir(agent.nn_dir) == ['last_stopped_custom_stop_ep_1.pth']


class _StatefulEnv:
    """what an env with state of its own adds to the discrete test env: get_env_state / set_env_state"""

    def __init__(self, env, state=None):
        self.env, self.state = env, state

    def __getattr__(self, name):
        return getattr(self.env, name)

    def get_env_state(self):
        return self.state

    def set_env_state(self, state):
        self.state = state


def test_discrete_checkpoint_carries_the_env_state(monkeypatch, tmp_path):
    a = _discrete(monkeypatch, tmp_path)
    a.vec_env = _StatefulEnv(a.vec_env, {'curriculum': 3})
    fn = str(tmp_path / 'ck')
    a.save(fn)
    b = _discrete(monkeypatch, tmp_path)
    b.vec_env = _StatefulEnv(b.vec_env)
    b.restore(fn + '.pth')
    assert b.vec_env.state == {'curriculum': 3}


def test_discrete_pbt_run_carries_its_index_in_the_experiment_name(monkeypatch, tmp_path):
    agent = _discrete(monkeypatch, tmp_path, over={'population_based_training': True, 'pbt_idx': 3})
    assert agent.experiment_name.startswith(agent.config['name'] + '_pbt_03_')
