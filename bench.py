"""bench.py -- PPO env-steps/s on the BASELINE.json workload, one JSON line on stdout (rank 0).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference algorithm on host cores

A "step" is one full PPO epoch (`agent.train_epoch()`: H-step rollout on the synthetic on-GPU env -> GAE ->
mini_epochs x num_minibatches updates) at BASELINE.json configs[1]: 16384 envs x horizon 16, obs 60, act 8,
MLP [256,128,64], minibatch 32768, 4 mini-epochs, hyper-parameters of configs/mujoco/ant_envpool.yaml.
N > 1 (torchrun): every rank owns its own 16384-env shard (weak scaling), one NCCL all-reduce of the flat
gradient (+KL slot) per minibatch; value = all ranks' env-steps / max-over-ranks device time.

Timing: W >= 3 warm-up epochs, then exactly K epochs, each bracketed by CUDA events on the launching stream,
L2 flushed (256 MiB write) between epochs outside the event pairs, barrier + synchronize on both sides of the
timed region, max over ranks.  nvidia-smi clocks are sampled during the timed region.

--dump-outputs DIR (B200 arm): after the timed epochs, rank 0 writes what the last one handed its caller -- the
per-minibatch losses, per-mini-epoch KLs and learning rate of train_epoch()'s tuple, and the model state it left --
as DIR/<name>.npy.  Every input is seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # a measurement writes nothing into the tree it runs from
_STDOUT = sys.stdout

WORKLOADS = {
    # BASELINE.json configs[1]
    'c2': dict(num_actors=16384, horizon=16, obs_dim=60, act_dim=8, units=[256, 128, 64], minibatch=32768, mini_epochs=4),
    # BASELINE.json configs[4] per-GPU shard (131072 envs / 8), obs 256, horizon 32
    'c5': dict(num_actors=16384, horizon=32, obs_dim=256, act_dim=8, units=[256, 128, 64], minibatch=32768, mini_epochs=4),
    # BASELINE.json configs[3]: Humanoid-shaped LSTM policy (obs 348, 17 actions, LSTM 256 before the MLP [512,256,128] of
    # configs/mujoco/humanoid_envpool.yaml, seq_length 4), 8192 envs -- BPTT minibatch path; every GEMM on the tensor cores (gemm_tc.cu),
    # cell / loss / optimiser kernels as on the fp32 path (--fp32: CUDA-core GEMMs)
    'c4': dict(num_actors=8192, horizon=32, obs_dim=348, act_dim=17, units=[512, 256, 128], minibatch=32768, mini_epochs=4,
               rnn_units=256, rnn_before_mlp=True, seq_length=4),
}
CONFIG_INDEX = {'c2': 1, 'c4': 3, 'c5': 4}


def make_params(w, device, env_name, multi_gpu, graph=True, seed=5, mixed_precision=True):
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': list(w['units']), 'activation': 'elu', 'initializer': {'name': 'default'}}}
    if w.get('rnn_units'):
        network['rnn'] = {'name': 'lstm', 'units': w['rnn_units'], 'layers': 1, 'before_mlp': w.get('rnn_before_mlp', True)}
    config = {'name': 'bench', 'env_name': env_name, 'reward_shaper': {'scale_value': 1.0}, 'device': device,
              'multi_gpu': multi_gpu, 'mixed_precision': mixed_precision, 'normalize_input': True, 'normalize_value': True,
              'value_bootstrap': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95, 'learning_rate': 3e-4,
              'lr_schedule': 'adaptive', 'kl_threshold': 0.008, 'grad_norm': 1.0, 'entropy_coef': 0.0, 'truncate_grads': True,
              'e_clip': 0.2, 'clip_value': True, 'use_smooth_clamp': True, 'bound_loss_type': 'regularisation',
              'bounds_loss_coef': 0.0, 'max_epochs': -1, 'num_actors': w['num_actors'], 'horizon_length': w['horizon'],
              'minibatch_size': w['minibatch'], 'mini_epochs': w['mini_epochs'], 'critic_coef': 2, 'print_stats': False,
              'train_dir': train_dir(), 'b200_cuda_graph': graph,
              'env_config': {'obs_dim': w['obs_dim'], 'act_dim': w['act_dim'], 'device': device, 'seed': seed}}
    if w.get('seq_length'):
        config['seq_length'] = w['seq_length']
    config.update(CFG_OVERRIDES)     # --cfg key=value: developer A/B switches (b200_* options), recorded in the JSON line
    return {'seed': seed, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'},
            'network': network, 'config': config}


CFG_OVERRIDES = {}
TRAIN_DIR = None
MAX_DUMP_BYTES = 64 << 20


def train_dir():
    """The agents' train_dir (checkpoints, summaries): a private temporary directory per process, removed at exit, so that a run
    writes nothing into the tree and runs by different users on one machine cannot collide."""
    global TRAIN_DIR
    if TRAIN_DIR is None:
        TRAIN_DIR = tempfile.mkdtemp(prefix='b200_bench_')
        atexit.register(shutil.rmtree, TRAIN_DIR, True)
    return TRAIN_DIR


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(',')])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 8]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        sm = sorted(float(r[1]) for r in rows)
        reasons = []
        for i, name in ((4, 'hw_slowdown'), (5, 'hw_thermal_slowdown'), (6, 'sw_thermal_slowdown'), (7, 'sw_power_cap')):
            if any(r[i].lower().startswith('active') for r in rows):
                reasons.append(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(rows[0][2]), 'reasons': reasons, 'samples': len(rows)}


def dist_info():
    return int(os.getenv('RANK', '0')), int(os.getenv('LOCAL_RANK', '0')), int(os.getenv('WORLD_SIZE', '1'))


# ===================================================================================== reference arm (CPU)
def run_cpu_oracle(w, steps, warmup, sample_envs):
    """The reference algorithm (oracle/ppo_oracle.py: plain-PyTorch restatement pinned to the real reference by
    tests/golden) on the host cores, all threads.  Returns (env_steps_per_s, ms_per_step, cores)."""
    from oracle import ppo_oracle as O
    cores = pick_cpu_threads(w)
    torch.set_num_threads(cores)
    N = sample_envs
    mb = max(w['horizon'], w['minibatch'] * N // w['num_actors'])
    env = O.SyntheticEnvCPU(N, w['obs_dim'], w['act_dim'], seed=5)
    params = O.init_params(w['obs_dim'], w['units'], w['act_dim'], seed=5)
    ag = O.OracleAgent(env, params, w['obs_dim'], w['act_dim'], w['units'], N, w['horizon'], mb,
                       {'mini_epochs': w['mini_epochs']})
    ag.obs = ag.env_reset()
    g = torch.Generator().manual_seed(0)
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        noise = torch.randn(w['horizon'], N, w['act_dim'], generator=g)
        ag.train_epoch(noise)
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    total = sum(ts)
    return N * w['horizon'] * steps / total, 1e3 * total / steps, cores


def available_cpus():
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:   # cgroup v2 CPU quota of the container
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def pick_cpu_threads(w):
    """All the host threads the reference can USE: intra-op parallelism of small fp32 ops stops scaling (and then
    collapses) well before 128 threads, so probe a tiny epoch at a few thread counts up to the available CPUs and keep
    the fastest (the reference's own default is min(4, cores), torch_runner.py:217-225)."""
    from oracle import ppo_oracle as O
    avail = available_cpus()
    cands = sorted({c for c in (avail, 64, 32, 16, 8, 4) if c <= avail})
    best, best_t = cands[0], float('inf')
    g = torch.Generator().manual_seed(0)
    for c in cands:
        torch.set_num_threads(c)
        N = 1024
        ag = O.OracleAgent(O.SyntheticEnvCPU(N, w['obs_dim'], w['act_dim'], seed=5), O.init_params(w['obs_dim'], w['units'], w['act_dim'], seed=5),
                           w['obs_dim'], w['act_dim'], w['units'], N, w['horizon'], max(w['horizon'], N * w['horizon'] // 8),
                           {'mini_epochs': 1})
        ag.obs = ag.env_reset()
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            ag.train_epoch(torch.randn(w['horizon'], N, w['act_dim'], generator=g))
            ts.append(time.perf_counter() - t0)
        if ts[-1] < best_t:
            best, best_t = c, ts[-1]
    return best


def cpu_reference_leg(w, steps, warmup):
    """CPU arm: the UNMODIFIED reference (oracle/_ref, vendored by __graft_entry__.build(); oracle/ref_arm.py) at the FULL workload
    shape when it is present, else the oracle port on a quarter-size sample.  Returns (value, ms, cpu_baseline dict)."""
    from oracle import ref_arm
    if ref_arm.available():
        cores = ref_arm.pick_threads(w, available_cpus())
        val, ms, play, upd = ref_arm.run_train_epochs(w, steps, warmup, cores)
        return val, ms, {'value': val, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'reference',
                         'sample': f'{steps} epochs after {warmup} warm-up of the unmodified reference A2CAgent.train_epoch() (rl_games @ oracle/_ref, '
                                   f'device cpu, fp32, torch_compile off, _pytorch_gae) at the full shape: {w["num_actors"]} envs x horizon '
                                   f'{w["horizon"]}, minibatch {w["minibatch"]} x {w["mini_epochs"]} mini-epochs',
                         'same_config': True, 'play_time_s': play, 'update_time_s': upd}
    sample = min(w['num_actors'], 4096)
    val, ms, cores = run_cpu_oracle(w, steps, warmup, sample)
    return val, ms, {'value': val, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port', 'same_config': False,
                     'sample': f'{sample} of {w["num_actors"]} envs per step, same horizon / mini-epochs / minibatch count; '
                               f'oracle/ppo_oracle.py (oracle/_ref absent on this box: port pinned by golden vectors)'}


def reference_arm(args, w):
    rank, _, world = dist_info()
    if rank != 0:
        return
    val, ms, cb = cpu_reference_leg(w, args.steps, max(1, args.warmup))
    line = {'impl': 'reference', 'metric': 'ppo_env_steps_per_sec', 'value': val, 'unit': 'env-steps/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args.workload, w, 'cpu synthetic env (oracle.ref_arm.SyntheticVecEnvCPU)'),
            'cpu_baseline': cb,
            'e2e': {'value': val, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), file=_STDOUT, flush=True)


def workload_config(name, w, env_desc):
    return {'workload': f'{name}: synthetic PPO, {w["num_actors"]} envs/GPU x horizon {w["horizon"]}, obs {w["obs_dim"]}, '
                        f'act {w["act_dim"]}, MLP {w["units"]}, minibatch {w["minibatch"]} x {w["mini_epochs"]} mini-epochs '
                        f'{"LSTM " + str(w["rnn_units"]) + " before the MLP, seq_length " + str(w["seq_length"]) + " " if w.get("rnn_units") else ""}'
                        f'(BASELINE.json configs[{CONFIG_INDEX[name]}])',
            'env': env_desc, 'global_batch': w['num_actors'] * w['horizon'], 'parallelism': 'dp (actors sharded per GPU)',
            'l2': 'flushed between steps (256 MiB write outside the per-step CUDA-event pairs)',
            'hyper_params': 'rl_games/configs/mujoco/ant_envpool.yaml:28-56'}


# ===================================================================================== B200 arm
def build_agent(w, device, env_name, multi_gpu, graph=True, mixed_precision=True):
    from rl_games_b200.runner import Runner
    r = Runner()
    r.load({'params': make_params(w, device, env_name, multi_gpu, graph, mixed_precision=mixed_precision)})
    agent = r.algo_factory.create(r.algo_name, base_name='bench', params=r.params)
    agent.init_tensors()
    agent.obs = agent.env_reset()
    return agent


def timed_epochs(agent, steps, flush, world):
    """Runs `steps` epochs; returns (ms per epoch, what the last train_epoch() returned)."""
    import torch.distributed as dist
    from rl_games_b200 import ops
    evs, result = [], None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    for _ in range(steps):
        if flush is not None:
            ops.fill_u32(flush, 1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        agent.epoch_num += 1
        result = agent.train_epoch()
        e.record()
        evs.append((s, e))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    return [s.elapsed_time(e) for s, e in evs], result


def dump_outputs(out_dir, agent, result):
    """Writes train_epoch()'s returned statistics (a_losses, c_losses, b_losses, entropies: one value per minibatch update; kls: one per
    mini-epoch; last_lr) and the model state it left (model.<state_dict key>) as float32 / float64 .npy files."""
    import numpy as np
    _, _, _, _, a_losses, c_losses, b_losses, entropies, kls, last_lr, _ = result
    arrays = {k: torch.stack([torch.as_tensor(x, dtype=torch.float32) for x in v]).numpy()
              for k, v in (('a_losses', a_losses), ('c_losses', c_losses), ('b_losses', b_losses), ('entropies', entropies), ('kls', kls))
              if len(v)}
    arrays['last_lr'] = np.array([last_lr], dtype=np.float64)
    for k, v in agent.model.state_dict().items():
        v = v.detach().cpu()          # fp64 normaliser moments and integer counts stay exact in float64
        arrays['model.' + k] = (v.double() if v.dtype == torch.float64 or not v.is_floating_point() else v.float()).numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > MAX_DUMP_BYTES:
        raise SystemExit(f'bench.py: --dump-outputs would write {total} bytes (limit {MAX_DUMP_BYTES})')
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def kernel_breakdown(agent):
    """One instrumented eager epoch: CUDA events around every C-ABI call -> per-kernel time shares + launch count."""
    from rl_games_b200._lib import lib
    graph = agent.use_cuda_graph
    agent.use_cuda_graph = False
    lib.start_profile()
    agent.epoch_num += 1
    agent.train_epoch()
    prof = lib.stop_profile()
    agent.use_cuda_graph = graph
    return prof


def gae_roofline(w, peaks):
    from rl_games_b200 import ops
    H, N = w['horizon'], w['num_actors']
    dev = torch.device('cuda', torch.cuda.current_device())
    r, v = torch.randn(H, N, device=dev), torch.randn(H, N, device=dev)
    d = (torch.rand(H, N, device=dev) < 0.05).to(torch.uint8)
    lv, ld = torch.randn(N, device=dev), (torch.rand(N, device=dev) < 0.05).to(torch.uint8)
    advs, rets = torch.empty(H, N, device=dev), torch.empty(H, N, device=dev)
    part = torch.zeros((N + 63) // 64, 8, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, cold, n=13):
        """cold: one launch per event pair behind an L2 flush (256 MiB write; the launch is enqueued while the flush still runs, so no CPU
        launch latency is inside the pair); not cold: 20 back-to-back launches inside one pair / 20 (L2-resident inputs, launch latency
        overlapped: what the kernel costs inside the epoch graph)"""
        ts = []
        for i in range(n):
            ops.fill_u32(flush if cold else flush[:1 << 20], 1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(1 if cold else 20):
                fn()
            e.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(s.elapsed_time(e) / (1 if cold else 20))
        return sum(ts) / len(ts)
    ours = lambda: ops.gae_fused(r, v, d, lv, ld, None, advs, rets, part, 0.99, 0.95)   # noqa: E731
    ms, ms_warm = timed(ours, True), timed(ours, False)
    alg = 17 * H * N + 8 * N     # r4 + V4 + done1 read, A4 + returns4 written per element; last_value/last_done per env
    gbs = alg / (ms * 1e-3) / 1e9
    try:
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get('gae_fused_f32')
    except Exception:
        tr = None
    out = {'kernel': 'gae_tma_kernel (GAE + returns + moment partials, TMA-staged)', 'bound': 'hbm', 'achieved': gbs,
           'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'], 'traffic': tr['traffic'] if tr else None,
           'alg_bytes_per_launch': alg, 'ms_per_launch': ms, 'ms_per_launch_l2_resident': ms_warm, 'peak_source': peaks['source'],
           'note': 'workload shape (4.5 MB working set, one launch ~ one DRAM round trip: latency bound; cold = L2 flushed before each launch, '
                   'l2_resident = what the kernel sees inside the epoch graph); large-shape asymptote and the comparators at every '
                   'shape: profiles/r02_gae_sweep.json (tools/gae_sweep.py)'}
    # the reference's own Triton kernel on the same box, same shape, same timing (gae_kernel.py:16-59 via _triton_gae), fp32 dones like its caller
    try:
        from oracle import ref_arm
        ref_arm.import_reference()
        from rl_games.triton_kernels.gae_kernel import _triton_gae
        r3, v3, lv2, df, ldf = r.unsqueeze(2), v.unsqueeze(2), lv.unsqueeze(1), d.float(), ld.float()
        tfn = lambda: _triton_gae(r3, v3, df, lv2, ldf, 0.99, 0.95)   # noqa: E731
        tfn()
        tms, tms_warm = timed(tfn, True), timed(tfn, False)
        out['reference_triton'] = {'kernel': 'rl_games.triton_kernels.gae_kernel._gae_kernel (advantages only, 16 B/element)', 'ms_per_launch': tms,
                                   'ms_per_launch_l2_resident': tms_warm, 'GBs': 16 * H * N / (tms * 1e-3) / 1e9,
                                   'speedup_cold': tms / ms, 'speedup_l2_resident': tms_warm / ms_warm}
    except Exception as e:
        out['reference_triton'] = {'unavailable': repr(e)[:200]}
    return out


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return {'hbm_gbs': j['hbm_gbs'], 'bf16_tflops': j['bf16_tflops'], 'bf16_tflops_sustained': j['bf16_tflops_sustained'],
                'source': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


def b200_arm(args, w):
    import torch.distributed as dist
    rank, local_rank, world = dist_info()
    multi = world > 1
    torch.cuda.set_device(local_rank)
    device = f'cuda:{local_rank}'
    peaks = load_peaks()
    agent = build_agent(w, device, 'b200_synthetic', multi, graph=not args.no_graph, mixed_precision=not args.fp32)
    if multi:
        dist.broadcast(agent.model.flat, 0)
        agent._repack()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    W = max(3, args.warmup)
    timed_epochs(agent, W, flush, world)
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    ms, result = timed_epochs(agent, args.steps, flush, world)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, agent, result)
    total_ms = torch.tensor([sum(ms)], dtype=torch.float64, device=device)
    if multi:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms) * 1e-3
    B = w['num_actors'] * w['horizon']
    value = B * world * args.steps / total_s
    # ---- kernel breakdown + launch count (instrumented eager epoch, not part of the timed region) ----
    prof = kernel_breakdown(agent)
    ktot = sum(v['ms'] for v in prof.values()) or 1.0
    kernels = sorted(({'call': k, 'launches': v['n'], 'ms': round(v['ms'], 4), 'share': round(v['ms'] / ktot, 4)}
                      for k, v in prof.items()), key=lambda x: -x['ms'])
    launches_per_step = sum(v['n'] for v in prof.values())
    line = {'metric': 'ppo_env_steps_per_sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': W, 'ms_per_step': 1e3 * total_s / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32' if args.fp32 else 'bf16', 'data': 'synthetic',
            'config': workload_config(args.workload, w, 'b200_synthetic (on-GPU Philox env, one kernel per step)'),
            'clocks': clocks, 'gpu_launches': launches_per_step * args.steps, 'gpu_launches_per_step': launches_per_step,
            'cuda_graph': ('whole-epoch' if agent._graph_epoch is not None else ('update-phase' if agent._graph_update is not None else 'none')), 'kernels': kernels[:12]}
    if CFG_OVERRIDES:
        line['config']['overrides'] = dict(CFG_OVERRIDES)
    if rank == 0:
        # dominant kernel family of the step -> roofline
        line['roofline_gae'] = gae_roofline(w, peaks)
        mlp_ms = sum(v['ms'] for k, v in prof.items() if 'linear' in k or 'tc_mlp' in k)       # linear_* covers the _f32 and the _tc GEMMs
        mlp_in = w.get('rnn_units') or w['obs_dim']
        flops = 2 * sum(a * b for a, b in zip([mlp_in] + w['units'], w['units'] + [w['act_dim'] + 1]))
        if w.get('rnn_units'):          # LSTM gate GEMMs: [obs + hidden] x 4 hidden per row
            flops += 2 * (w['obs_dim'] + w['rnn_units']) * 4 * w['rnn_units']
        step_flops = B * flops * (1 + 1.0 / w['horizon'] + 3 * w['mini_epochs'])   # rollout fwd (+ last-value fwd) + (fwd + dgrad + wgrad) per mini-epoch
        tf = step_flops / (mlp_ms * 1e-3) / 1e12 if mlp_ms > 0 else 0.0
        fam = ('MLP / LSTM GEMM kernels: fp32 CUDA-core path (mixed_precision: False)' if args.fp32 else
               'layer-wise bf16 tcgen05 GEMMs (gemm_tc_kernel<fwd|dgrad|wgrad>: LSTM gates + MLP)' if w.get('rnn_units') else
               'tcgen05 bf16 MLP kernels (mlp_fwd_tc<train|rollout>, mlp_bwd_tc)')
        family = {'kernels': fam, 'bound': 'tensor', 'achieved': tf, 'peak': peaks['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                  'frac': tf / peaks['bf16_tflops_sustained'], 'share_of_step': round(mlp_ms / ktot, 4), 'alg_flops_per_step': step_flops}
        # the single dominant kernel of the step (largest share of device time): algorithmic FLOPs per launch / its mean launch
        # duration (CUDA events around each launch of the instrumented epoch); `traffic` = DRAM bytes per launch from the
        # committed ncu --set full capture (profiles/traffic.json), null when that kernel has no capture
        dims = list(zip([mlp_in] + w['units'], w['units'] + [w['act_dim'] + 1]))
        fwd_fl = 2 * sum(a * b for a, b in dims)
        dgrad_fl = 2 * sum(a * b for a, b in dims[1:])           # no input gradient for the first layer
        per_launch = {'tc_mlp_bwd': (fwd_fl + dgrad_fl) * w['minibatch'], 'tc_mlp_fwd_train': fwd_fl * w['minibatch'],
                      'tc_mlp_fwd_rollout': fwd_fl * w['num_actors']}
        dom = max((k for k in prof if k in per_launch), key=lambda k: prof[k]['ms'], default=None)
        if dom is not None:
            dms = prof[dom]['ms'] / prof[dom]['n']
            dtf = per_launch[dom] / (dms * 1e-3) / 1e12
            try:
                tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get(dom)
            except Exception:
                tr = None
            line['roofline'] = {'kernel': dom, 'bound': 'tensor', 'achieved': dtf, 'peak': peaks['bf16_tflops_sustained'],
                                'unit': 'TFLOP/s', 'frac': dtf / peaks['bf16_tflops_sustained'],
                                'traffic': tr['traffic'] if tr else None, 'traffic_source': tr['source'] if tr else None,
                                'alg_flops_per_launch': per_launch[dom], 'ms_per_launch': dms,
                                'share_of_step': round(prof[dom]['ms'] / ktot, 4), 'peak_source': peaks['source'] + ' bf16 sustained',
                                'family': family,
                                'note': 'K = 60..256, N = 16..256 GEMMs fused with their elementwise epilogues (ELU, bf16 pack, loss, '
                                        'delta chain): bound by epilogue latency / MMA issue, far below the dense-GEMM peak by '
                                        'construction; stage timelines in profiles/r01_stage_timing.md'}
        else:
            line['roofline'] = dict(family, kernel=fam, traffic=None, peak_source=peaks['source'] + ' bf16 sustained')
        if world == 1 and not args.skip_e2e:
            line['e2e'] = e2e_leg(w, device, args)
        if world == 1 and not args.skip_cpu:
            _, _, line['cpu_baseline'] = cpu_reference_leg(w, 3, 1)
    # ---- second workload on the same line: BASELINE configs[4]'s per-GPU shard (obs 256, horizon 32) -- the shape the multi-GPU
    #      north_star names -- so that the driver's 1/2/4/8-GPU runs carry its curve too (same timing protocol, all ranks)
    if args.workload == 'c2' and not args.skip_secondary:
        agent._graph_update = agent._graph_epoch = None
        del agent
        torch.cuda.synchronize()
        w5 = WORKLOADS['c5']
        agent = build_agent(w5, device, 'b200_synthetic', multi, graph=not args.no_graph, mixed_precision=not args.fp32)
        if multi:
            dist.broadcast(agent.model.flat, 0)
            agent._repack()
        timed_epochs(agent, 3, flush, world)
        k5 = max(3, min(args.steps, 10))
        ms5, _ = timed_epochs(agent, k5, flush, world)
        t5 = torch.tensor([sum(ms5)], dtype=torch.float64, device=device)
        if multi:
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
        if rank == 0:
            t5s = float(t5) * 1e-3
            line['c5'] = {'metric': 'ppo_env_steps_per_sec', 'value': w5['num_actors'] * w5['horizon'] * world * k5 / t5s, 'unit': 'env-steps/s',
                          'n_gpus': world, 'steps': k5, 'warmup': 3, 'ms_per_step': 1e3 * t5s / k5, 'scaling': 'weak', 'dtype': line['dtype'],
                          'config': workload_config('c5', w5, 'b200_synthetic (on-GPU Philox env, one kernel per step)'),
                          'kernels': 'l1_fwd_tc + mlp_fwd_tc<XL1> / l1_wgrad_tc + mlp_bwd_tc<XL1> (wide-observation tcgen05 path)'}
    if rank == 0:
        print(json.dumps(line), file=_STDOUT, flush=True)
    if multi:
        # drop captured graphs (they hold NCCL kernels) before tearing the communicator down; NCCL teardown at interpreter
        # exit can hang with captured collectives alive, so leave with a hard exit once everything is flushed
        agent._graph_update = agent._graph_epoch = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stderr.flush()
        _STDOUT.flush()
        shutil.rmtree(train_dir(), ignore_errors=True)      # os._exit skips the atexit removal
        os._exit(0)


def e2e_leg(w, device, args):
    """Same metric through the public API with a HOST env: every env step copies obs/rewards/dones/time-outs
    host->device (pinned) and the actions device->host; the per-epoch stats block is read back."""
    agent = build_agent(w, device, 'b200_synthetic_host', False, graph=not args.no_graph, mixed_precision=not args.fp32)
    K = max(3, min(args.steps, 10))
    for _ in range(3):
        agent.epoch_num += 1
        agent.train_epoch()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        agent.epoch_num += 1
        agent.train_epoch()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    N, H, D, A = w['num_actors'], w['horizon'], w['obs_dim'], w['act_dim']
    h2d = H * (N * D * 4 + N * 4 + N + N)
    d2h = H * N * A * 4 + agent.stats.numel() * 4 + 10 * 8
    return {'value': N * H * K / dt, 'unit': 'env-steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
            'steps': K, 'env': 'b200_synthetic_host (numpy env in host memory, pinned staging, wall-clock timed)'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='c2', choices=list(WORKLOADS))
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--fp32', action='store_true', help='mixed_precision: False (fp32 CUDA-core MLP kernels)')
    ap.add_argument('--cfg', action='append', default=[], help='config override key=value (python literal), e.g. b200_pipelined_wgrad=False')
    ap.add_argument('--skip-e2e', action='store_true')
    ap.add_argument('--skip-cpu', action='store_true')
    ap.add_argument('--skip-secondary', action='store_true', help='do not append the c5 block to the c2 line')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed epoch returned and the model state it left as DIR/<name>.npy (B200 arm)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to the B200 arm')
    w = WORKLOADS[args.workload]
    import ast
    for kv in args.cfg:
        k, v = kv.split('=', 1)
        CFG_OVERRIDES[k] = ast.literal_eval(v)
    # stdout carries exactly ONE JSON line: everything else (Runner's seed banner etc.) goes to stderr
    import contextlib
    global _STDOUT
    _STDOUT = sys.stdout
    with contextlib.redirect_stdout(sys.stderr):
        if args.impl == 'reference':
            reference_arm(args, w)
            return
        if not torch.cuda.is_available():
            raise SystemExit('bench.py: the B200 arm needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
        b200_arm(args, w)


if __name__ == '__main__':
    main()
