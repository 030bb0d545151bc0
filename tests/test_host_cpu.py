"""CPU-only tests: the C-ABI library loads and exports every symbol include/b200rl.h declares (no compute calls without
a GPU), host-side config logic / error behaviour mirrors the reference, and the multi-GPU host logic works over a real
2-process `gloo` group (the reference's own strategy: tests/test_multigpu_stats_sync.py:80-115)."""
import ctypes
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ppo_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from rl_games_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos) >= 30 and 'b200rl_gae_f32' in protos and 'b200rl_tc_mlp_bwd' in protos
    assert os.path.exists(_lib.LIB_PATH), 'build with __graft_entry__.build() first'
    cdll = ctypes.CDLL(_lib.LIB_PATH)
    for name in protos:
        assert hasattr(cdll, name), f'{name} declared in include/b200rl.h but not exported'
    assert _lib.lib.b200rl_version() >= 100 and _lib.lib.b200rl_built_arch() == 100
    # pure host-side queries are safe without a GPU
    assert _lib.lib.b200rl_tc_supported(60, 256, 128, 64, 8) == 1
    assert _lib.lib.b200rl_tc_supported(348, 256, 128, 64, 17) == 0
    assert _lib.lib.b200rl_loss_partial_stride() == 40


def test_product_library_exports_exactly_the_header_and_no_test_hooks():
    """include/b200rl.h IS the export list: nothing undeclared leaves the product library; the test-only host entry points
    (b200rl_hosttest_*, `#ifdef B200RL_TEST_HOOKS`) live in tests/libb200rl_testhooks.so, which nothing under rl_games_b200/ loads"""
    import subprocess
    from rl_games_b200 import _lib
    from tests import _hooks

    def exported(path):
        out = subprocess.run(['nm', '-D', '--defined-only', path], capture_output=True, text=True, check=True).stdout
        return {ln.split()[-1] for ln in out.splitlines() if ' T ' in ln and ln.split()[-1].startswith('b200rl_')}
    declared = set(_lib.parse_header())
    assert exported(_lib.LIB_PATH) == declared
    _hooks.load()
    extra = exported(_hooks.HOOKS_LIB_PATH) - declared
    assert extra and all(n.startswith('b200rl_hosttest_') for n in extra), extra
    for root, _, files in os.walk(os.path.join(ROOT, 'rl_games_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(root, f)).read()
                if f != 'build.py':      # only the build script names the test library
                    assert 'testhooks' not in src and 'hosttest' not in src, f


def test_header_prototypes_parse_types():
    from rl_games_b200 import _lib
    p = _lib.parse_header()
    sig = dict(p['b200rl_gae_f32'])
    assert sig['gamma'] is ctypes.c_double and sig['H'] is ctypes.c_int and sig['r_st_t'] is ctypes.c_int64
    assert sig['stream'] is ctypes.c_void_p and sig['rewards'] is ctypes.c_void_p
    assert dict(p['b200rl_synth_env_step'])['seed'] is ctypes.c_uint64


def test_ops_refuse_cpu_tensors_no_fallback():
    from rl_games_b200 import ops
    r = torch.zeros(4, 3, 1)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.compute_gae(r, r, torch.zeros(4, 3), torch.zeros(3, 1), torch.zeros(3), 0.99, 0.95)


def _params(**over):
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': [16, 8], 'activation': 'elu', 'initializer': {'name': 'default'}}}
    from rl_games_b200.common import Box
    config = {'name': 't', 'env_name': 'unused', 'reward_shaper': {'scale_value': 1.0}, 'device': 'cpu', 'normalize_input': True,
              'normalize_value': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95, 'learning_rate': 3e-4,
              'lr_schedule': 'adaptive', 'kl_threshold': 0.008, 'grad_norm': 1.0, 'entropy_coef': 0.0, 'e_clip': 0.2, 'clip_value': True,
              'num_actors': 8, 'horizon_length': 8, 'minibatch_size': 32, 'mini_epochs': 2, 'critic_coef': 2,
              'env_info': {'observation_space': Box(-1, 1, (6,)), 'action_space': Box(-1, 1, (3,))}}
    config.update(over)
    return {'seed': 1, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'}, 'network': network, 'config': config}


def test_agent_has_no_cpu_fallback_and_mirrors_config_errors(tmp_path):
    from rl_games_b200.runner import Runner
    r = Runner()
    r.load({'params': _params(train_dir=str(tmp_path))})
    assert r.algo_name == 'a2c_continuous' and r.seed == 1
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        r.algo_factory.create(r.algo_name, base_name='x', params=r.params)
    with pytest.raises(ValueError):
        r.algo_factory.create('sac', base_name='x', params=r.params)            # ObjectFactory: unknown name -> ValueError(name)
    r2 = Runner()
    r2.load({'params': _params(train_dir=str(tmp_path), multi_gpu_sync_stats_mode='bogus')})
    with pytest.raises(ValueError, match='multi_gpu_sync_stats_mode'):             # a2c_common.py:99-103
        r2.algo_factory.create(r2.algo_name, base_name='x', params=r2.params)


def test_schedulers_match_reference_golden():
    from rl_games_b200.common import AdaptiveScheduler, LinearScheduler
    m = torch.load(os.path.join(ROOT, 'tests', 'golden', 'math.pt'), weights_only=False)
    sch, lr = AdaptiveScheduler(0.008), 3e-4
    for k, ref in zip(m['adaptive']['kls'], m['adaptive']['lrs']):
        lr, _ = sch.update(lr, 0.0, 0, 0, k)
        assert lr == ref
    lin = LinearScheduler(1e-3, min_lr=1e-6, max_steps=100)
    assert lin.update(0, 0, 50, 0, 0)[0] == pytest.approx(1e-6 + (1e-3 - 1e-6) * 0.5, rel=1e-12)   # tests/test_critical_fixes.py:89-115


def test_gae_c_oracle_matches_torch_oracle_bitexact():
    lib_path = os.path.join(ROOT, 'oracle', '_build', 'libgae_oracle.so')
    if not os.path.exists(lib_path):
        pytest.skip('oracle/_build not built (run __graft_entry__.build())')
    lib = ctypes.CDLL(lib_path)
    g = torch.Generator().manual_seed(0)
    H, N = 16, 33
    r, v = torch.randn(H, N, generator=g), torch.randn(H, N, generator=g)
    d = (torch.rand(H, N, generator=g) < 0.15).float()
    lv, ld = torch.randn(N, generator=g), (torch.rand(N, generator=g) < 0.15).float()
    out = torch.empty(H, N)
    lib.gae_oracle_f32(*(ctypes.c_void_p(t.data_ptr()) for t in (r, v, d, lv, ld, out)), H, N, ctypes.c_double(0.99), ctypes.c_double(0.95))
    ref = O.gae(r.unsqueeze(2), v.unsqueeze(2), d, lv.unsqueeze(1), ld, 0.99, 0.95).squeeze(2)
    assert torch.equal(out, ref)


# ------------------------------------------------------------------------------------------ 2-process gloo
def _worker(rank, world, port, ret):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from rl_games_b200.dist_utils import merge_stats_packed
    g = torch.Generator().manual_seed(100 + rank)
    # --- pooled running-stat merge: two normalisers in ONE packed all-reduce, two epochs of deltas ---
    D = 5
    rms = [O.RunningMeanStd((D,)), O.RunningMeanStd((1,))]
    snaps = {}
    data = [[], []]
    for epoch in range(2):
        for i, m in enumerate(rms):
            x = torch.randn(40 + 10 * rank, D if i == 0 else 1, generator=g) * (1 + i) + rank
            data[i].append(x)
            m.train(); m(x); m.eval()
        mods = [(f'm{i}', m.count.reshape(1), m.running_mean, m.running_var) for i, m in enumerate(rms)]
        snaps = merge_stats_packed(mods, snaps, lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM))
        for i, m in enumerate(rms):
            m.count = mods[i][1].reshape(())
    # gather every rank's raw data to check against the pooled moments
    out = {}
    for i in range(2):
        mine = torch.cat(data[i])
        sizes = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([mine.shape[0]]))
        mx = int(max(s.item() for s in sizes))
        pad = torch.zeros(mx, mine.shape[1]); pad[:mine.shape[0]] = mine
        bufs = [torch.zeros_like(pad) for _ in range(world)]
        dist.all_gather(bufs, pad)
        allx = torch.cat([b[:int(s)] for b, s in zip(bufs, sizes)]).double()
        n = allx.shape[0] + world      # every rank starts with the count=1 prior (mean 0, var 1)
        out[i] = (int(rms[i].count), n, rms[i].running_mean.clone(), allx.sum(0) / n,
                  rms[i].running_var.clone(), ((allx ** 2).sum(0) + world * 1.0) / n - (allx.sum(0) / n) ** 2)
    # --- flat gradient + KL slot all-reduce (a2c_common.py:493-509 + :1559-1561) ---
    P = 11
    comm = torch.arange(P + 1, dtype=torch.float32) * (rank + 1)
    dist.all_reduce(comm, op=dist.ReduceOp.SUM)
    ret[rank] = (out, comm / world)
    dist.barrier()
    dist.destroy_process_group()


def test_two_process_gloo_stats_merge_and_grad_allreduce():
    world, port = 2, 29000 + os.getpid() % 1000
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    for i in range(2):
        (c0, n0, m0, em0, v0, ev0), (c1, n1, m1, em1, v1, ev1) = ret[0][0][i], ret[1][0][i]
        assert c0 == c1 == n0
        assert torch.equal(m0, m1) and torch.equal(v0, v1)                      # byte-identical across ranks after the merge
        torch.testing.assert_close(m0, em0, rtol=1e-6, atol=1e-6)              # == pooled moments of all data (+ priors); batch moments are fp32 (reference tolerance 1e-5)
        torch.testing.assert_close(v0, ev0, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(ret[0][1], torch.arange(12, dtype=torch.float32) * 1.5)
    assert torch.equal(ret[0][1], ret[1][1])


def test_merge_matches_reference_merge_rank_stats_with_fake_allreduce():
    """tests/test_multigpu_stats_sync.py:14-17 strategy: an injected all-reduce that models two identical ranks."""
    from rl_games_b200.dist_utils import merge_stats_packed
    g = torch.Generator().manual_seed(3)
    m = O.RunningMeanStd((4,))
    m.train(); m(torch.randn(50, 4, generator=g) * 2 + 1); m.eval()
    ref = O.RunningMeanStd((4,)); ref.load(m.state())
    snap_ref = O.merge_rank_stats(ref, lambda t: t.mul_(2))
    mods = [('obs', m.count.reshape(1), m.running_mean, m.running_var)]
    snaps = merge_stats_packed(mods, {}, lambda t: t.mul_(2))
    assert int(mods[0][1]) == int(ref.count)
    torch.testing.assert_close(m.running_mean, ref.running_mean, rtol=1e-12, atol=0)
    torch.testing.assert_close(m.running_var, ref.running_var, rtol=1e-12, atol=1e-15)
    for a, b in zip(snaps['obs'], snap_ref):
        torch.testing.assert_close(a.reshape(-1), b.reshape(-1).double(), rtol=1e-12, atol=0)


def test_reference_checkpoint_wire_format_roundtrip(monkeypatch):
    """SURVEY 8f rank 3: a checkpoint dict written by the REAL reference (tests/golden/gen_golden.py checkpoint:
    A2CBase.get_full_state_weights after one epoch) loads into the flat-arena model and re-exports with the same keys, the same
    key ORDER (players index `model` by name, torch.optim.Adam.load_state_dict indexes parameters by position) and identical
    tensors -- weights, normaliser statistics, Adam moments, step and lr.  Pure host logic: runs on CPU tensors."""
    import torch
    from rl_games_b200 import ops
    from rl_games_b200.model import B200Model
    # the fp32 mirror of the normaliser statistics is refreshed by a CUDA kernel; irrelevant for the key/tensor mapping under test
    monkeypatch.setattr(ops, 'refresh_norm', lambda *a, **k: None)
    g = torch.load(os.path.join(os.path.dirname(__file__), 'golden', 'ref_checkpoint.pt'), weights_only=False)
    ck = g['checkpoint']
    net = {'name': 'actor_critic', 'separate': False,
           'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                    'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
           'mlp': {'units': g['units'], 'activation': 'elu', 'initializer': {'name': 'default'}}}
    m = B200Model(net, g['D'], g['A'], 'cpu', normalize_input=True, normalize_value=True, seed=1)
    m.load_state_dict(ck['model'])
    lr, step = m.load_optimizer_state_dict(ck['optimizer'])
    sd = m.state_dict()
    assert list(sd.keys()) == list(ck['model'].keys())
    for k, v in ck['model'].items():
        assert sd[k].dtype == v.dtype, k
        assert torch.equal(sd[k].reshape(v.shape), v), k
    ref_opt = ck['optimizer']
    assert lr == ref_opt['param_groups'][0]['lr'] and step == int(ref_opt['state'][0]['step'])
    osd = m.optimizer_state_dict(lr, step, ref_opt['param_groups'][0]['weight_decay'])
    assert osd['param_groups'][0]['params'] == ref_opt['param_groups'][0]['params']
    for key in ('lr', 'betas', 'eps', 'weight_decay', 'amsgrad'):
        assert osd['param_groups'][0][key] == ref_opt['param_groups'][0][key], key
    assert sorted(osd['state'].keys()) == sorted(ref_opt['state'].keys())
    names = g['param_order']          # reference model.parameters() order == the optimizer's positional order
    for i, name in enumerate(names):
        for f in ('exp_avg', 'exp_avg_sq'):
            assert torch.equal(osd['state'][i][f].reshape(ref_opt['state'][i][f].shape), ref_opt['state'][i][f]), (name, f)
        assert float(osd['state'][i]['step']) == float(ref_opt['state'][i]['step'])
        assert osd['state'][i]['exp_avg'].numel() == ck['model'][name].numel(), name


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly ONE JSON line on stdout with the keys of
    the bench contract, a cpu_baseline block describing the run and an e2e block that repeats the line's own value."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
              'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['metric'] == 'ppo_env_steps_per_sec' and d['unit'] == 'env-steps/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 1 and d['warmup'] == 1 and 'workload' in d['config']
    assert d['cpu_baseline']['kind'] in ('port', 'reference') and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


@pytest.mark.parametrize('patch,what', [({'normalization': 'layer_norm'}, 'normalization'), ({'name': 'resnet_actor_critic'}, 'resnet_actor_critic'),
                                        ({'mlp': {'units': [16, 8], 'activation': 'elu', 'initializer': {'name': 'default'}, 'd2rl': True}}, 'd2rl'),
                                        ({'separate': True, 'rnn': {'name': 'lstm', 'units': 8, 'layers': 1}}, 'separate actor/critic trunks with an rnn'),
                                        ({'joint_obs_actions': {}}, 'joint_obs_actions')])
def test_network_options_without_a_kernel_fail_loudly(patch, what):
    """a config option that changes the network's maths (network_builder.py:545-589) is either implemented or refused -- never ignored"""
    from rl_games_b200.model import B200Model
    net = {'name': 'actor_critic', 'separate': False,
           'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                    'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
           'mlp': {'units': [16, 8], 'activation': 'elu', 'initializer': {'name': 'default'}, 'regularizer': {'name': 'l2_regularizer'}}}
    net.update(patch)
    with pytest.raises(NotImplementedError, match=what):
        B200Model(net, 6, 3, 'cpu', True, True)


def test_index_less_cuda_device_resolves_to_the_current_device(monkeypatch):
    """`device: cuda` (configs/ppo_cartpole.yaml = BASELINE configs[0], ppo_lunar_discrete.yaml): the reference hands the string to torch, which
    resolves it to the current device; here raw pointers cross the C ABI and torch.cuda.set_device refuses an index-less device, so the agents
    make the index explicit.  'cuda:N' and non-CUDA names pass through untouched (the latter are refused by the agents: no CPU fallback)."""
    from rl_games_b200.model import resolve_device
    monkeypatch.setattr(torch.cuda, 'current_device', lambda: 3)
    assert resolve_device('cuda') == torch.device('cuda', 3)
    assert resolve_device('cuda:1') == torch.device('cuda', 1) and resolve_device(torch.device('cuda:0')) == torch.device('cuda', 0)
    assert resolve_device('cpu') == torch.device('cpu')
    seen = []
    monkeypatch.setattr(torch.cuda, 'set_device', lambda d: seen.append(d))
    from rl_games_b200 import agent_discrete
    stub = type('A', (), {'ppo_device': 'cuda', '_require_cuda': agent_discrete.DiscreteA2CAgent._require_cuda})()
    stub._require_cuda()
    assert seen == [torch.device('cuda', 3)]
