"""TEST / BASELINE INFRASTRUCTURE ONLY -- never imported by the product path (rl_games_b200/).

The UNMODIFIED reference (Denys88/rl_games) as the CPU arm of bench.py (`--impl reference`, `cpu_baseline.kind:
"reference"`) and as the on-GPU Triton-GAE comparator (tools/gae_sweep.py).

* vendor(): the reference is pure Python and its build backend (hatchling) is not in this image, so
  `pip install --target` cannot run offline; what a wheel install would do -- place the `rl_games/` package tree,
  byte for byte, on a path -- is done directly: /root/reference/rl_games -> oracle/_ref/rl_games.  oracle/_ref/ is
  git-ignored (never in history) but not gpurun-ignored, so it travels to the GPU box, where /root/reference does not
  exist.  Called from __graft_entry__.build() in the build container.
* the two packages the reference imports that this image lacks (gymnasium, tensorboardX) come from the import stubs
  under tests/golden/_stubs (shape/dtype descriptors and a no-op writer; no arithmetic).
* run_train_epochs(): BASELINE.md section 4 protocol -- `A2CAgent.train_epoch()` (a2c_common.py:1517-1584) built through
  `Runner.algo_factory` with the env injected via config['env_info'] / config['vec_env'] (a2c_common.py:236-241),
  device cpu, mixed_precision False, torch_compile False, compute_gae -> _pytorch_gae (gae_kernel.py:62-79, :139).
"""
import atexit
import hashlib
import json
import os
import shutil
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_SRC = '/root/reference'
REF_DST = os.path.join(HERE, '_ref')
STUBS = os.path.join(ROOT, 'tests', 'golden', '_stubs')
_TRAIN_DIR = None


def _tree_digest(path):
    h = hashlib.sha256()
    for dp, dn, fn in sorted(os.walk(path)):
        dn.sort()
        for f in sorted(fn):
            if f.endswith('.pyc'):
                continue
            p = os.path.join(dp, f)
            h.update(os.path.relpath(p, path).encode())
            with open(p, 'rb') as fh:
                h.update(fh.read())
    return h.hexdigest()


def vendor(verbose=True):
    """Copy the reference package tree verbatim into oracle/_ref/ (build container only).  Returns True if available."""
    src = os.path.join(REF_SRC, 'rl_games')
    dst = os.path.join(REF_DST, 'rl_games')
    meta_p = os.path.join(REF_DST, 'VENDORED.json')
    if not os.path.isdir(src):
        return os.path.isdir(dst)
    digest = _tree_digest(src)
    if os.path.isdir(dst) and os.path.exists(meta_p):
        try:
            if json.load(open(meta_p)).get('sha256') == digest and _tree_digest(dst) == digest:
                return True
        except Exception:
            pass
    shutil.rmtree(dst, ignore_errors=True)
    os.makedirs(REF_DST, exist_ok=True)
    shutil.copytree(src, dst, ignore=shutil.ignore_patterns('__pycache__', '*.pyc'))
    for extra in ('LICENSE',):
        if os.path.exists(os.path.join(REF_SRC, extra)):
            shutil.copy(os.path.join(REF_SRC, extra), os.path.join(REF_DST, extra))
    json.dump({'source': src, 'sha256': digest, 'how': 'verbatim copytree of the pure-Python package (hatchling absent: pip cannot build offline)'},
              open(meta_p, 'w'))
    if verbose:
        print(f'oracle/_ref: vendored the unmodified reference package ({digest[:12]})')
    return True


def available():
    return os.path.isdir(os.path.join(REF_DST, 'rl_games'))


def import_reference():
    """Put the stubs + the vendored reference on sys.path and import it.  Raises ImportError when it was never vendored."""
    if not available():
        raise ImportError('oracle/_ref/rl_games is missing: run __graft_entry__.build() in the build container')
    for p in (STUBS, REF_DST):
        if p not in sys.path:
            sys.path.insert(0, p)
    import rl_games  # noqa: F401
    return rl_games


class SyntheticVecEnvCPU:
    """BASELINE.md section 4 synthetic env on the host (same distribution as the on-GPU env of the B200 arm): obs ~ N(0,1), reward
    -||a||^2, done at t >= 100 or with p = 0.01, time_outs on the t >= 100 subset.  Tensor env -> the reference's tensor path."""

    def __init__(self, num_envs, obs_dim, act_dim, seed=5, max_len=100, p_done=0.01):
        import torch
        self.N, self.D, self.A = num_envs, obs_dim, act_dim
        self.g = torch.Generator().manual_seed(seed)
        self.max_len, self.p_done = max_len, p_done
        self.t = torch.zeros(num_envs, dtype=torch.int32)

    def reset(self):
        import torch
        self.t.zero_()
        return torch.randn(self.N, self.D, generator=self.g)

    def step(self, actions):
        import torch
        rew = -(actions * actions).sum(-1)
        self.t += 1
        time_out = self.t >= self.max_len
        term = torch.rand(self.N, generator=self.g) < self.p_done
        done = time_out | term
        self.t[done] = 0
        obs = torch.randn(self.N, self.D, generator=self.g)
        return obs, rew, done.to(torch.uint8), {'time_outs': time_out & ~term}

    def get_env_info(self):
        import numpy as np
        import gymnasium as gym
        return {'observation_space': gym.spaces.Box(-np.inf, np.inf, (self.D,), np.float32),
                'action_space': gym.spaces.Box(-1.0, 1.0, (self.A,), np.float32)}

    def get_env_state(self):
        return None

    def set_env_state(self, s):
        pass

    def set_train_info(self, *a, **kw):
        pass


def _train_dir():
    """The reference agents' train_dir: private to this process and removed at exit, so runs by different users cannot collide."""
    global _TRAIN_DIR
    if _TRAIN_DIR is None:
        _TRAIN_DIR = tempfile.mkdtemp(prefix='b200_refarm_')
        atexit.register(shutil.rmtree, _TRAIN_DIR, True)
    return _TRAIN_DIR


def make_params(w, num_actors, minibatch, mini_epochs=None):
    """c2 / c5 hyper-parameters (rl_games/configs/mujoco/ant_envpool.yaml:28-56), the same dict bench.py gives the B200 arm."""
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': list(w['units']), 'activation': 'elu', 'initializer': {'name': 'default'}}}
    if w.get('rnn_units'):
        network['rnn'] = {'name': 'lstm', 'units': w['rnn_units'], 'layers': 1, 'before_mlp': w.get('rnn_before_mlp', False)}
    config = {'name': 'refarm', 'env_name': 'unused', 'reward_shaper': {'scale_value': 1.0}, 'device': 'cpu', 'multi_gpu': False,
              'mixed_precision': False, 'torch_compile': False, 'normalize_input': True, 'normalize_value': True,
              'value_bootstrap': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95, 'learning_rate': 3e-4,
              'lr_schedule': 'adaptive', 'kl_threshold': 0.008, 'grad_norm': 1.0, 'entropy_coef': 0.0, 'truncate_grads': True,
              'e_clip': 0.2, 'clip_value': True, 'use_smooth_clamp': True, 'bound_loss_type': 'regularisation',
              'bounds_loss_coef': 0.0, 'max_epochs': -1, 'num_actors': num_actors, 'horizon_length': w['horizon'],
              'minibatch_size': minibatch, 'mini_epochs': mini_epochs or w['mini_epochs'], 'critic_coef': 2, 'save_frequency': 0,
              'save_best_after': 10 ** 9, 'print_stats': False, 'train_dir': _train_dir()}
    if w.get('seq_length'):
        config['seq_length'] = w['seq_length']
    return {'seed': 5, 'torch_threads': 0, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'},
            'network': network, 'config': config}


def build_reference_agent(w, num_actors=None, minibatch=None, mini_epochs=None):
    """The reference's own A2CAgent on the host, env injected (tests/test_ppo_masking.py:92-107 pattern)."""
    import_reference()
    from rl_games.torch_runner import Runner
    N = num_actors or w['num_actors']
    mb = minibatch or w['minibatch']
    env = SyntheticVecEnvCPU(N, w['obs_dim'], w['act_dim'], seed=5)
    params = make_params(w, N, mb, mini_epochs)
    params['config']['env_info'] = env.get_env_info()
    runner = Runner()
    runner.load({'params': params})
    runner.params['config']['vec_env'] = env
    agent = runner.algo_factory.create(runner.algo_name, base_name='refarm', params=runner.params)
    agent.init_tensors()
    agent.obs = agent.env_reset()
    return agent


def pick_threads(w, avail):
    """All the host threads the reference can USE: probe a small epoch at a few thread counts and keep the fastest (its own default
    is min(4, cores), torch_runner.py:217-225; intra-op scaling of these small fp32 ops stops well before 100+ threads)."""
    import torch
    cands = sorted({c for c in (avail, 64, 32, 16, 8, 4) if c <= avail})
    best, best_t = cands[0], float('inf')
    for c in cands:
        torch.set_num_threads(c)
        N = 2048
        ag = build_reference_agent(w, num_actors=N, minibatch=N * w['horizon'] // 4, mini_epochs=1)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            ag.train_epoch()
            ts.append(time.perf_counter() - t0)
        if ts[-1] < best_t:
            best, best_t = c, ts[-1]
    return best


def run_train_epochs(w, steps, warmup, threads):
    """Times `steps` reference train_epoch() calls at the FULL workload shape after `warmup`.  Returns (env_steps_per_s, ms_per_step,
    play_time_s, update_time_s) -- the last two are the reference's own split (a2c_common.py:1583)."""
    import torch
    torch.set_num_threads(threads)
    ag = build_reference_agent(w)
    ts, play, upd = [], 0.0, 0.0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = ag.train_epoch()
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
            play += out[1]
            upd += out[2]
    total = sum(ts)
    return w['num_actors'] * w['horizon'] * steps / total, 1e3 * total / steps, play / steps, upd / steps


if __name__ == '__main__':
    print('vendored:', vendor())
