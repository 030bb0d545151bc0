"""bench.py's B200 arm end to end without a GPU (tests/_bench_dryrun.py: recorder library, no compute): the measurement script must
get from the command line to ONE JSON line carrying the contract keys whatever the host changes of the round were."""
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
KEYS = ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
        'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline')


@pytest.mark.parametrize('extra', [[], ['--workload', 'c5'], ['--fp32'], ['--workload', 'c4']])
def test_bench_b200_arm_reaches_its_json_line(extra):
    r = subprocess.run([sys.executable, os.path.join(HERE, '_bench_dryrun.py'), '--steps', '2', '--warmup', '1', '--no-graph', '--skip-cpu'] + extra,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    out = json.loads(lines[0])
    for k in KEYS:
        assert k in out, k
    assert out['metric'] == 'ppo_env_steps_per_sec' and out['n_gpus'] == 1 and out['steps'] == 2 and out['warmup'] >= 3
    fp32 = '--fp32' in extra
    assert out['dtype'] == ('f32' if fp32 else 'bf16')
    assert set(out['e2e']) >= {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'}
    assert ('c5' in out['config']['workload']) == ('c5' in extra)
    if not extra:       # the default (c2) line also carries BASELINE configs[4]'s per-GPU shard
        assert out['c5']['n_gpus'] == 1 and out['c5']['value'] > 0 and 'obs 256' in out['c5']['config']['workload']
    rec = json.loads([ln for ln in r.stderr.splitlines() if ln.startswith('RECORDED ')][-1][len('RECORDED '):])
    if 'c4' in extra:       # LSTM policy: gate / MLP GEMMs on the tensor cores layer by layer, cell kernels as on the fp32 path
        assert rec['b200rl_lstm_cell_fwd_f32'] > 0 and rec['b200rl_lstm_cell_bwd_f32'] > 0 and 'LSTM 256' in out['config']['workload']
        assert rec['b200rl_linear_fwd_tc'] > 0 and rec['b200rl_linear_bwd_weight_tc'] > 0 and 'b200rl_linear_fwd_f32' not in rec
    elif fp32:
        assert 'b200rl_ppo_head_loss_f32' in rec and 'b200rl_tc_mlp_fwd_train' not in rec
    else:
        assert rec['b200rl_tc_mlp_fwd_train'] > 0 and rec['b200rl_tc_mlp_bwd'] > 0 and rec['b200rl_synth_env_step'] > 0


def test_bench_steps_sets_the_timed_epochs_and_dump_outputs_writes_the_last_one(tmp_path):
    """--steps K runs exactly K more epochs (H env steps each); --dump-outputs DIR writes train_epoch()'s returned statistics and the model
    state as float32 / float64 .npy files, within 64 MB"""
    import numpy as np
    env_steps = {}
    for k in (1, 3):
        r = subprocess.run([sys.executable, os.path.join(HERE, '_bench_dryrun.py'), '--steps', str(k), '--warmup', '1', '--no-graph', '--skip-cpu',
                            '--skip-e2e', '--skip-secondary', '--dump-outputs', str(tmp_path / f'k{k}')], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout)['steps'] == k
        env_steps[k] = json.loads([ln for ln in r.stderr.splitlines() if ln.startswith('RECORDED ')][-1][len('RECORDED '):])['b200rl_synth_env_step']
    assert env_steps[3] - env_steps[1] == 2 * 16                 # c2: horizon 16
    d = tmp_path / 'k3'
    out = {f[:-len('.npy')]: np.load(d / f) for f in os.listdir(d)}
    n_upd = 4 * (16384 * 16 // 32768)                             # c2: mini-epochs x minibatches per mini-epoch
    for k in ('a_losses', 'c_losses', 'b_losses', 'entropies'):
        assert out[k].shape == (n_upd,), k
    assert out['kls'].shape == (4,) and out['last_lr'].shape == (1,)
    assert out['model.a2c_network.actor_mlp.0.weight'].shape == (256, 60) and out['model.a2c_network.mu.weight'].shape == (8, 64)
    assert out['model.running_mean_std.running_mean'].dtype == np.float64
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    r = subprocess.run([sys.executable, os.path.join(HERE, '_bench_dryrun.py'), '--steps', '0'], capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and '--steps' in r.stderr
