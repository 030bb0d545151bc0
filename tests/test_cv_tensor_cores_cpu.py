"""Host logic of the tensor-core critic (central_value_config mixed_precision: True) without a GPU: precision routing, the golden run of
tests/golden/agent_cv.pt with torch stand-ins for the tensor-core GEMMs and the fused value head, the refresh of the critic's bf16 weight
twin, and the C-ABI calls an mjlab config makes through the reference's Runner.  The kernels themselves are checked on a B200 in
tests/test_cv_tensor_cores_gpu.py."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _torch_ops as T  # noqa: E402
import test_agent_cv_host_cpu as HC  # noqa: E402

GOLDEN = os.path.join(HERE, 'golden')


# ---------------------------------------------------------------------------------------------- stand-ins for the two new ops
def value_head_loss(a_last, W_v, b_v, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count, act_last,
                    d_alast, dW_part, db_part, split_stride, n_splits, partials, value_out=None):
    """b200rl_value_head_loss_f32 restated: the value GEMV, the value-loss stand-in, d(a_last) and the head gradient (all of it in split 0)"""
    al = a_last[:M]
    v = (al @ W_v.reshape(-1) + b_v).unsqueeze(1)
    dv = torch.zeros(M, 1)
    nb = T.value_loss(v, 1, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count, dv, 1, partials)
    d_alast[:M] = (dv * W_v.reshape(1, -1)) * T._act_grad_from_out(al, act_last)
    fw, fb = T._flat(dW_part), T._flat(db_part)
    Hl = W_v.numel()
    for s in range(n_splits):
        fw[s * split_stride:s * split_stride + Hl] = (dv * al).sum(0) if s == 0 else 0.0
        fb[s * split_stride] = dv.sum() if s == 0 else 0.0
    if value_out is not None:
        value_out[:M] = v.squeeze(1)
    return nb


def value_head_fwd(a_last, W_v, b_v, vms_mean, vms_var, normalize_value, values, N):
    v = a_last[:N] @ W_v.reshape(-1) + b_v
    values.copy_(T.normalize(v, vms_mean, vms_var, denorm=True) if normalize_value else v)


def _install_value_head(monkeypatch):
    from rl_games_b200 import ops
    monkeypatch.setattr(ops, 'value_head_loss', value_head_loss)
    monkeypatch.setattr(ops, 'value_head_fwd', value_head_fwd)


def _golden(mp):
    """agent_cv.pt with the critic's precision key set to mp (None: absent)"""
    g = dict(torch.load(os.path.join(GOLDEN, 'agent_cv.pt'), weights_only=False))
    cv = dict(g['cv_config'])
    cv.pop('mixed_precision', None)
    if mp is not None:
        cv['mixed_precision'] = mp
    g['cv_config'] = cv
    return g


# ---------------------------------------------------------------------------------------------- routing
@pytest.mark.parametrize('mp', [True, False, None], ids=['true', 'false', 'absent'])
def test_the_critic_precision_comes_from_its_own_key(mp, monkeypatch, tmp_path, capsys):
    """central_value_config.mixed_precision decides (True -> tensor cores; False / absent -> fp32, absent with a note); the agent-level key
    does not: it is set to the opposite of the critic's here"""
    _install_value_head(monkeypatch)
    agent = HC._build_cv(monkeypatch, tmp_path, _golden(mp), over={'mixed_precision': not mp})
    cv = agent.central_value_net
    assert cv.gemm_tc is bool(mp)
    assert cv.n_splits == (max(1, min(16, cv.minibatch_size // 512)) if mp else max(1, min(64, cv.minibatch_size // 256)))
    assert hasattr(cv, 'wbf') is bool(mp)
    note = 'central_value_config.mixed_precision not set' in capsys.readouterr().out
    assert note is (mp is None)


def test_a_last_layer_wider_than_the_fused_head_takes_is_refused(monkeypatch, tmp_path):
    from rl_games_b200 import ops
    g = _golden(True)
    g['cv_units'] = [8, ops.VALUE_HEAD_MAX_HL + 1]
    with pytest.raises(NotImplementedError, match='fused value head'):
        HC._build_cv(monkeypatch, tmp_path, g)


# ---------------------------------------------------------------------------------------------- golden run on stand-ins
def test_tensor_core_critic_host_logic_matches_reference_golden(monkeypatch, tmp_path):
    """the whole golden comparison of test_agent_cv_host_cpu (same tolerances), with the critic on the tensor-core route: every trunk GEMM
    through the *_tc stand-ins, the value head through the fused-head stand-ins, and never the fp32 value-loss op"""
    from rl_games_b200 import ops
    _install_value_head(monkeypatch)
    calls = {}

    def count(name, f):
        def g(*a, **k):
            calls[name] = calls.get(name, 0) + 1
            return f(*a, **k)
        return g
    built = []
    build = HC._build_cv

    def build_tc(mp_, tmp, g, over=None):
        built.append(build(mp_, tmp, {**g, 'cv_config': {**g['cv_config'], 'mixed_precision': True}}, over))
        for n in ('value_head_loss', 'value_head_fwd', 'value_loss', 'linear_fwd_tc', 'linear_bwd_weight_tc'):     # after the stand-ins
            mp_.setattr(ops, n, count(n, getattr(ops, n)))
        return built[-1]
    monkeypatch.setattr(HC, '_build_cv', build_tc)
    HC.test_central_value_agent_host_logic_matches_reference_golden(False, monkeypatch, tmp_path)
    cv = built[0].central_value_net
    assert cv.gemm_tc
    n_mb = cv.mini_epoch * cv.num_minibatches * len(torch.load(os.path.join(GOLDEN, 'agent_cv.pt'), weights_only=False)['epochs_out'])
    assert calls['value_head_loss'] == n_mb and calls.get('value_loss', 0) == 0
    assert calls['value_head_fwd'] >= cv.H and calls['linear_fwd_tc'] > 0 and calls['linear_bwd_weight_tc'] >= n_mb * len(cv.units)


# ---------------------------------------------------------------------------------------------- the bf16 twin
def test_the_twin_is_refreshed_after_every_critic_step_and_every_load(monkeypatch, tmp_path):
    """a spy on cast_bf16: one refresh of the critic's arena follows every critic Adam step before the next critic GEMM, and each of the
    four load paths refreshes it"""
    from rl_games_b200 import ops
    from rl_games_b200 import runner as R
    _install_value_head(monkeypatch)
    g = _golden(True)
    a = HC._build_cv(monkeypatch, tmp_path, g)
    cv = a.central_value_net
    log = []
    cast, adam, fwd = ops.cast_bf16, ops.adam_step, ops.linear_fwd_tc

    def spy_cast(src, dst):
        log.append(('cast', src.data_ptr() == cv.flat.data_ptr() and dst.data_ptr() == cv.wbf.data_ptr()))
        cast(src, dst)

    def spy_adam(params, *x, **k):
        log.append(('adam', params.data_ptr() == cv.flat.data_ptr()))
        adam(params, *x, **k)

    def spy_fwd(X, W, *x, bf16_arena=None, **k):
        log.append(('gemm', bf16_arena is not None and bf16_arena[1].data_ptr() == cv.wbf.data_ptr()))
        fwd(X, W, *x, bf16_arena=bf16_arena, **k)
    monkeypatch.setattr(ops, 'cast_bf16', spy_cast)
    monkeypatch.setattr(ops, 'adam_step', spy_adam)
    monkeypatch.setattr(ops, 'linear_fwd_tc', spy_fwd)
    flat_noise = g['noise'].reshape(-1, g['N'], g['A'])
    a.epoch_num += 1
    a.train_epoch(noise=flat_noise[:g['H']])
    steps = [i for i, e in enumerate(log) if e == ('adam', True)]
    assert len(steps) == cv.mini_epoch * cv.num_minibatches
    for i in steps:
        nxt = [e for e in log[i + 1:] if e in (('cast', True), ('gemm', True))]
        assert nxt and nxt[0] == ('cast', True), 'a critic GEMM ran on a stale twin'
    a.save(str(tmp_path / 'ck'))
    ck = torch.load(str(tmp_path / 'ck.pth'), weights_only=False)

    def refreshes(fn):
        n0 = log.count(('cast', True))
        fn()
        return log.count(('cast', True)) - n0
    assert refreshes(lambda: cv.load_state_dict(ck['assymetric_vf_nets'])) >= 1
    assert refreshes(lambda: a.set_full_state_weights(ck)) >= 1
    assert refreshes(lambda: a.set_central_value_function_weights(ck)) >= 1
    assert refreshes(lambda: R._restore(a, {'train': True, 'checkpoint': str(tmp_path / 'ck.pth'), 'load_critic_only': True})) >= 1


def test_rollout_values_follow_loaded_weights_through_the_twin(monkeypatch, tmp_path):
    """stand-ins that, like the kernels, read the weights from the bf16 twin: after a critic-only load, get_value is the forward of the
    LOADED weights (rounded to bf16), not of the ones the twin held before"""
    from rl_games_b200 import ops
    from rl_games_b200 import runner as R
    _install_value_head(monkeypatch)

    def twin_fwd(X, W, b, Y, act, bf16_arena=None, **k):
        flat, fb = bf16_arena
        o = (W.data_ptr() - flat.data_ptr()) // 4
        T.linear_fwd(X, fb[o:o + W.numel()].view(W.shape).float(), b, Y, act, **k)
    g = _golden(True)
    a = HC._build_cv(monkeypatch, tmp_path, g)
    flat_noise = g['noise'].reshape(-1, g['N'], g['A'])
    a.epoch_num += 1
    a.train_epoch(noise=flat_noise[:g['H']])
    a.save(str(tmp_path / 'ck'))
    b = HC._build_cv(monkeypatch, tmp_path, g)
    monkeypatch.setattr(ops, 'linear_fwd_tc', twin_fwd)
    cvb = b.central_value_net
    states = g['state_tape'][0].clone()
    before = torch.zeros(g['N'])
    cvb.get_value(states, before)
    R._restore(b, {'train': True, 'checkpoint': str(tmp_path / 'ck.pth'), 'load_critic_only': True})
    got = torch.zeros(g['N'])
    cvb.get_value(states, got)
    ref = cvb.flat.clone()
    acts = [torch.zeros(g['N'], u) for u in cvb.units]
    r = cvb.running_mean_std
    x = states
    for i, u in enumerate(cvb.units):
        W = cvb.view(f'W{i}', ref).to(torch.bfloat16).float()
        T.linear_fwd(x, W, cvb.view(f'b{i}', ref), acts[i], cvb.act_id, norm_mean=r.mean_f32 if i == 0 else None,
                     norm_std=r.std_f32 if i == 0 else None)
        x = acts[i]
    want = torch.zeros(g['N'])
    value_head_fwd(x, cvb.view('W_v'), cvb.view('b_v'), cvb.value_mean_std.running_mean, cvb.value_mean_std.running_var, True, want, g['N'])
    torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-6)
    assert not torch.allclose(got, before, rtol=1e-3, atol=1e-4)


# ---------------------------------------------------------------------------------------------- the reference's Runner on an mjlab config
def test_mjlab_config_with_a_tensor_core_critic_runs_through_the_reference_runner(monkeypatch, tmp_path):
    """configs/mjlab/ppo_go1_velocity.yaml with central_value_config.mixed_precision: True injected (and nothing else but what a launcher
    sets): one epoch through the reference's Runner, every C-ABI call header-checked; the critic issues the tensor-core GEMMs and the
    fused value head, never the fp32 value loss"""
    import yaml
    import test_reference_runner_cpu as RR
    if RR.REF is None:
        pytest.skip('reference rl_games package not vendored into oracle/_ref')
    for p in (os.path.join(HERE, 'golden', '_stubs'), RR.REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from rl_games.torch_runner import Runner
    import rl_games_b200
    from rl_games_b200.agent_cv import A2CAgentCV
    rec = RR.ABI._patch(monkeypatch)
    cfg = yaml.safe_load(open(os.path.join(RR.REF, 'rl_games', 'configs', 'mjlab', 'ppo_go1_velocity.yaml')))
    c = cfg['params']['config']
    assert 'mixed_precision' not in c['central_value_config']
    c['central_value_config']['mixed_precision'] = True
    N = c['num_actors']
    D, A = RR._GENERIC_DIMS
    env = RR._GymEnvCV(N, D, RR._CV_STATE_DIM, A)
    c.update({'env_info': env.get_env_info(), 'vec_env': env, 'device': RR.H._CudaLookingStr('cpu'), 'max_epochs': 1, 'train_dir': str(tmp_path),
              'b200_cuda_graph': False, 'multi_gpu': False})
    c.pop('max_frames', None)
    runner = rl_games_b200.register(Runner())
    runner.load(cfg)
    runner.params['config']['vec_env'] = env
    made = []
    orig_create = runner.algo_factory.create
    monkeypatch.setattr(runner.algo_factory, 'create', lambda name, **kw: (made.append(orig_create(name, **kw)), made[-1])[1])
    runner.run({'train': True, 'play': False, 'checkpoint': None, 'sigma': None})
    agent, = made
    assert type(agent) is A2CAgentCV and agent.epoch_num == 1 and agent.central_value_net.gemm_tc
    assert not agent.gemm_tc and not agent.use_tc           # the actor's own key is absent: [512,256,128] stays on its fp32 kernels
    cv = agent.central_value_net
    n_cv = cv.mini_epoch * cv.num_minibatches
    assert rec.calls['b200rl_value_head_loss_f32'] == n_cv
    assert rec.calls['b200rl_value_head_fwd_f32'] == c['horizon_length'] + 1
    assert rec.calls['b200rl_linear_bwd_weight_tc'] == n_cv * len(cv.units)
    assert rec.calls['b200rl_linear_bwd_data_tc'] == n_cv * (len(cv.units) - 1)
    assert rec.calls['b200rl_linear_fwd_tc'] == (n_cv + c['horizon_length'] + 1) * len(cv.units)
    assert rec.calls['b200rl_cast_bf16'] >= n_cv + 1
    assert 'b200rl_value_loss_f32' not in rec.calls
