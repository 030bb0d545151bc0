"""INTEGRATION.md section 1 as a test: the B200 agent registered into the REFERENCE's own `rl_games.torch_runner.Runner`
(torch_runner.py:98-354), a stock YAML of the reference loaded unchanged (configs/mujoco/ant_envpool.yaml), `runner.run(...)`.

No GPU: every C-ABI call is answered by the header-checking recorder of test_abi_calls_cpu (argument count / ctypes types against
include/b200rl.h, returns success), so what is tested is the boundary -- the reference Runner's config injection (DefaultRewardsShaper
object, features.observer, seed handling), its run_train sequence (_restore, _override_sigma, torch.compile of agent.model: the stock
YAML leaves torch_compile at its default True) and the agent's train() loop with the reference's own DefaultAlgoObserver.
The reference is the verbatim copy of its package that __graft_entry__.build() places in oracle/_ref when the reference source is at hand;
without it these tests skip: the reference's Runner is code, not data, and the repository does not carry it."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import test_abi_calls_cpu as ABI  # noqa: E402
import test_agent_host_cpu as H  # noqa: E402

ROOT = os.path.dirname(HERE)


REF = os.path.join(ROOT, 'oracle', '_ref')
if not os.path.isdir(os.path.join(REF, 'rl_games')):
    REF = None
pytestmark = pytest.mark.skipif(REF is None, reason='reference rl_games package not vendored into oracle/_ref')


class _GymEnv:
    """what config['env_info'] / config['vec_env'] injection needs (a2c_common.py:236-241); spaces are the stub's gymnasium Boxes,
    i.e. what a reference user would pass"""

    def __init__(self, N, D, A):
        self.N, self.D, self.A = N, D, A

    def reset(self):
        return torch.zeros(self.N, self.D)

    def step(self, actions):
        assert tuple(actions.shape) == (self.N, self.A)
        z8 = torch.zeros(self.N, dtype=torch.uint8)
        return torch.zeros(self.N, self.D), torch.zeros(self.N), z8, {'time_outs': z8}

    def get_env_info(self):
        import gymnasium as gym
        import numpy as np
        return {'observation_space': gym.spaces.Box(-np.inf, np.inf, (self.D,), np.float32),
                'action_space': gym.spaces.Box(-1.0, 1.0, (self.A,), np.float32)}

    def set_train_info(self, *a, **kw):
        pass

    def get_env_state(self):
        return None

    def set_env_state(self, s):
        pass


@pytest.mark.parametrize('obs_dim', [27, 105])      # Ant without / with contact forces: resident-W1 and wide-observation tcgen05 kernels
def test_stock_yaml_trains_through_the_reference_runner(obs_dim, monkeypatch, tmp_path, capsys):
    import yaml
    for p in (os.path.join(HERE, 'golden', '_stubs'), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from rl_games.torch_runner import Runner
    from rl_games.common.algo_observer import DefaultAlgoObserver
    from rl_games_b200.agent import A2CAgent as B200A2CAgent

    rec = ABI._patch(monkeypatch)
    cfg = yaml.safe_load(open(os.path.join(REF, 'rl_games', 'configs', 'mujoco', 'ant_envpool.yaml')))
    c = cfg['params']['config']
    assert c['mixed_precision'] is True and 'torch_compile' not in c          # the YAML itself is untouched below except for:
    env = _GymEnv(c['num_actors'], obs_dim, 8)
    c.update({'env_info': env.get_env_info(), 'vec_env': env, 'device': H._CudaLookingStr('cpu'), 'max_epochs': 2,
              'train_dir': str(tmp_path), 'b200_cuda_graph': False})

    runner = Runner()
    runner.algo_factory.register_builder('a2c_continuous', lambda **kwargs: B200A2CAgent(**kwargs))      # INTEGRATION.md section 1
    runner.load(cfg)
    runner.params['config']['vec_env'] = env          # Runner.load deep-copies the config
    made = []
    orig_create = runner.algo_factory.create

    def create(name, **kw):
        a = orig_create(name, **kw)
        made.append(a)
        return a
    monkeypatch.setattr(runner.algo_factory, 'create', create)
    runner.run({'train': True, 'play': False, 'checkpoint': None, 'sigma': None})

    agent, = made
    assert isinstance(agent, B200A2CAgent) and isinstance(agent.algo_observer, DefaultAlgoObserver)
    assert type(agent.rewards_shaper).__module__.startswith('rl_games.')          # the reference's DefaultRewardsShaper object, accepted as is
    assert hasattr(agent.model, 'load_optimizer_state_dict')                       # torch.compile(agent.model) was ignored, not installed
    assert 'torch.compile of agent.model ignored' in capsys.readouterr().out
    assert agent.epoch_num == 2 and agent.frame == 2 * c['num_actors'] * c['horizon_length']
    assert agent.use_tc and agent.tc_wide == (obs_dim > 64)
    n_upd = 2 * c['mini_epochs'] * (c['num_actors'] * c['horizon_length'] // c['minibatch_size'])
    assert rec.calls['b200rl_tc_mlp_fwd_train'] == n_upd and rec.calls['b200rl_tc_mlp_bwd'] == n_upd
    assert rec.calls['b200rl_tc_mlp_fwd_rollout'] == 2 * (c['horizon_length'] + 1)
    assert rec.calls['b200rl_gae_fused_f32'] == 2
    ckpts = os.listdir(agent.nn_dir)
    assert any(f.startswith('last_Ant-v5_envpool_ep_2') and f.endswith('.pth') for f in ckpts), ckpts
    sd = torch.load(os.path.join(agent.nn_dir, ckpts[0]), weights_only=False)
    assert {'model', 'optimizer', 'epoch', 'frame', 'last_mean_rewards'} <= set(sd) and 'a2c_network.mu.weight' in sd['model']


# ---------------------------------------------------------------------------------------------------------------- every shipped PPO YAML
# Families whose PPO configs are single-agent, flat-observation tasks (the path this repo builds); atari / minigrid (CNN), smac / ma
# (multi-agent, self-play) are outside it by construction and are not listed.
_FAMILIES = ('.', 'dm_control', 'maniskill', 'mujoco', 'mjlab', 'pufferlib', 'test')
_DIMS = {'ant': (105, 8), 'halfcheetah': (17, 6), 'hopper': (11, 3), 'humanoid': (348, 17), 'walker2d': (17, 6)}       # Gymnasium v5 obs / act
_GENERIC_DIMS = (24, 6)             # the other tasks' YAMLs do not fix the env's dimensions
_CV_STATE_DIM = 30
# What is NOT built raises NotImplementedError at construction -- never a silent reinterpretation.  file -> the reason it gives:
_REFUSED = {
    'carracing_ppo.yaml': "'cnn' networks", 'maniskill/ppo_pick_cube_rgbd_NOT_WORKING_YET.yaml': "'cnn' networks",
    'ppo_cartpole_masked_velocity_rnn.yaml': "'rnn' networks are not supported by the discrete", 'test/test_rnn.yaml': "'rnn' networks are not supported by the discrete",
    'test/test_rnn_multidiscrete_mhv.yaml': "'rnn' networks are not supported by the discrete",
    'ppo_lunar_continiuos_torch.yaml': 'separate actor/critic trunks with an rnn', 'ppo_pendulum.yaml': 'state-dependent sigma',
    'test/test_asymmetric_continuous.yaml': 'separate actor/critic trunks with an rnn|rnn: only a single-layer',
    'ppo_continuous_lstm.yaml': "model 'continuous_a2c_lstm_logstd'", 'ppo_walker_rnn.yaml': "rnn: only a single-layer 'lstm'",
    'ppo_walker_tcnn.yaml': "network 'tcnnnet'", 'test/test_discrite_testnet_aux_loss.yaml': "network 'testnet_aux_loss'",
    'test/test_asymmetric_discrete.yaml': 'central_value_config|rnn', 'test/test_asymmetric_discrete_mhv.yaml': 'central_value_config',
    'test/test_asymmetric_discrete_mhv_mops.yaml': 'central_value_config|testnet', 'test/test_rnn_multidiscrete.yaml': 'central_value_config',
    # state-dependent sigma (fixed_sigma: false, softplus) and a minibatch (16384) that is not a whole number of envs' horizons (40)
    'mjlab/ppo_wujihand_reorient.yaml': 'minibatch_size must be a multiple of horizon_length|state-dependent sigma',
}
_MULTI_AGENT = {'ppo_multiwalker.yaml', 'ppo_smac.yaml'}          # multi-agent envs: refused by construction (test_host_cpu), need an env to say so


def _shipped_ppo_yamls():
    if REF is None:
        return []
    import yaml
    out = []
    base = os.path.join(REF, 'rl_games', 'configs')
    for fam in _FAMILIES:
        d = os.path.join(base, fam)
        if not os.path.isdir(d):
            continue
        for f in sorted(os.listdir(d)):
            rel = f if fam == '.' else os.path.join(fam, f)
            if not f.endswith('.yaml') or rel in _MULTI_AGENT:
                continue
            try:
                algo = yaml.safe_load(open(os.path.join(d, f)))['params']['algo']['name']
            except Exception:
                continue
            if algo in ('a2c_continuous', 'a2c_discrete'):
                out.append(rel)
    return out


class _GymEnvCV(_GymEnv):
    """tensor env with a privileged observation group (what rl_games' mjlab wrapper hands the agent: {'obs', 'states'} + state_space)"""

    def __init__(self, N, D, S, A):
        super().__init__(N, D, A)
        self.S = S

    def _o(self):
        return {'obs': torch.zeros(self.N, self.D), 'states': torch.zeros(self.N, self.S)}

    def reset(self):
        return self._o()

    def step(self, actions):
        _, r, d, info = super().step(actions)
        return self._o(), r, d, info

    def get_env_info(self):
        import gymnasium as gym
        import numpy as np
        info = super().get_env_info()
        info.update(state_space=gym.spaces.Box(-np.inf, np.inf, (self.S,), np.float32), use_global_observations=True)
        return info


class _GymEnvDiscrete(_GymEnv):
    def __init__(self, N, D, K):
        self.N, self.D, self.K = N, D, K

    def step(self, actions):
        z8 = torch.zeros(self.N, dtype=torch.uint8)
        return torch.zeros(self.N, self.D), torch.zeros(self.N), z8, {'time_outs': z8}

    def get_env_info(self):
        import gymnasium as gym
        import numpy as np
        space = gym.spaces.Discrete(self.K) if isinstance(self.K, int) else gym.spaces.Tuple([gym.spaces.Discrete(k) for k in self.K])
        return {'observation_space': gym.spaces.Box(-np.inf, np.inf, (self.D,), np.float32), 'action_space': space}


@pytest.mark.parametrize('rel', _shipped_ppo_yamls())
def test_every_shipped_ppo_yaml_of_the_in_scope_families_runs_through_the_reference_runner(rel, monkeypatch, tmp_path):
    """`rl_games_b200.register(runner)` into the reference's own Runner, then EVERY PPO YAML the reference ships for single-agent
    flat-observation tasks -- MuJoCo (Gymnasium / envpool / Ray back-ends), dm_control, ManiSkill, pufferlib, mjlab (central value +
    `schedule_type: standard` + `algo_observer: isaac`), the top-level and test configs -- UNCHANGED: only what a launcher injects is set
    (`env_info` / `vec_env`, `device`, `max_epochs`, `train_dir`, single process).  Each one either trains (one epoch of `runner.run`, every
    C-ABI call header-checked, the right agent class, the kernel family its geometry selects, the reference's own observer objects driving our
    agent) or is in `_REFUSED` and raises NotImplementedError with the listed reason."""
    import yaml
    for p in (os.path.join(HERE, 'golden', '_stubs'), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from rl_games.torch_runner import Runner
    import rl_games.common.algo_observer as ref_obs
    import rl_games_b200
    from rl_games_b200 import agent_discrete
    from rl_games_b200.agent import A2CAgent
    from rl_games_b200.agent_cv import A2CAgentCV

    rec = ABI._patch(monkeypatch)
    monkeypatch.setattr(agent_discrete.DiscreteA2CAgent, '_require_cuda', lambda self: None)
    monkeypatch.setattr(agent_discrete.DiscreteA2CAgent, '_sync', staticmethod(lambda: None))
    cfg = yaml.safe_load(open(os.path.join(REF, 'rl_games', 'configs', rel)))
    c, net = cfg['params']['config'], cfg['params']['network']
    discrete = cfg['params']['algo']['name'] == 'a2c_discrete'
    cv = bool(c.get('central_value_config'))
    N = c['num_actors']
    D, A = _DIMS.get(os.path.basename(rel).split('_')[0].split('.')[0], _GENERIC_DIMS) if rel.startswith('mujoco') else _GENERIC_DIMS
    if discrete:
        env = _GymEnvDiscrete(N, 12, [3, 4] if 'multi_discrete' in net.get('space', {}) else 4)
    elif cv:
        env = _GymEnvCV(N, D, _CV_STATE_DIM, A)
    else:
        env = _GymEnv(N, D, A)
    c.update({'env_info': env.get_env_info(), 'vec_env': env, 'device': 'cpu' if discrete else H._CudaLookingStr('cpu'), 'max_epochs': 1,
              'train_dir': str(tmp_path), 'b200_cuda_graph': False, 'multi_gpu': False})
    c.pop('max_frames', None)
    runner = Runner()
    assert rl_games_b200.register(runner) is runner
    runner.load(cfg)
    runner.params['config']['vec_env'] = env
    made = []
    orig_create = runner.algo_factory.create
    monkeypatch.setattr(runner.algo_factory, 'create', lambda name, **kw: (made.append(orig_create(name, **kw)), made[-1])[1])
    if rel in _REFUSED:
        with pytest.raises(NotImplementedError, match=_REFUSED[rel]):
            runner.run({'train': True, 'play': False, 'checkpoint': None, 'sigma': None})
        return
    runner.run({'train': True, 'play': False, 'checkpoint': None, 'sigma': None})
    agent, = made
    assert agent.epoch_num == 1 and agent.frame == N * c['horizon_length']
    assert isinstance(agent.algo_observer, ref_obs.IsaacAlgoObserver if c.get('algo_observer') == 'isaac' else ref_obs.DefaultAlgoObserver)
    if discrete:
        assert type(agent) is agent_discrete.DiscreteA2CAgent and rec.calls['b200rl_categorical_loss_f32'] > 0
        return
    assert type(agent) is (A2CAgentCV if cv else A2CAgent) and agent.has_central_value == cv
    assert agent.model.min_sigma == net['space']['continuous'].get('min_sigma', 0.0)
    units = net['mlp']['units']
    separate = bool(net.get('separate', False))          # two trunks = one block-structured MLP of twice the width, never on the fused kernels
    assert agent.model.separate == separate and agent.model.trunk_units == units and agent.model.units == [u * (2 if separate else 1) for u in units]
    fused = len(units) == 3 and all(u <= m for u, m in zip(units, (256, 128, 64))) and 'rnn' not in net and agent.model.min_sigma == 0 \
        and net['mlp']['activation'] in ('elu', 'relu', 'tanh') and not separate
    mp = c.get('mixed_precision')
    mb = c.get('minibatch_size') or N * c['minibatch_size_per_env']
    n_upd = c['mini_epochs'] * (N * c['horizon_length'] // mb)
    if fused and mp is not False:                                        # absent key = auto -> fused tcgen05 kernels where the geometry has them
        assert agent.use_tc and rec.calls['b200rl_tc_mlp_fwd_train'] == n_upd and rec.calls['b200rl_tc_mlp_bwd'] == n_upd
    elif mp is True:                                                     # e.g. [512,256,128] with mixed_precision: True -> layer-wise tcgen05 GEMMs
        assert agent.gemm_tc and rec.calls['b200rl_linear_fwd_tc'] > 0 and rec.calls['b200rl_linear_bwd_weight_tc'] >= n_upd * (len(units) + 1)
        assert rec.calls.get('b200rl_linear_fwd_f32', 0) == 0
    else:                                                                # key absent on such a geometry -> fp32 kernels (a printed note says so)
        assert not agent.use_tc and not agent.gemm_tc and rec.calls['b200rl_linear_bwd_weight_f32'] >= n_upd * (len(units) + 1)
    if cv:
        assert agent.schedule_type == c.get('schedule_type', 'per_minibatch') and rec.calls['b200rl_value_loss_f32'] > 0


def test_env_registered_in_the_reference_registries_is_built_without_injection(monkeypatch, tmp_path):
    """No `vec_env` / `env_info` injection: the YAML names an env that is registered only in the REFERENCE's registries
    (rl_games.common.vecenv.register + env_configurations.register, what envpool / gymnasium / user plugins do); the agent, running under the
    reference's Runner, builds it through those registries (common/vecenv.py:379-391) and reads its spaces from `get_env_info()`."""
    import yaml
    for p in (os.path.join(HERE, 'golden', '_stubs'), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from rl_games.torch_runner import Runner
    from rl_games.common import vecenv, env_configurations
    import rl_games_b200
    from rl_games_b200 import common as C

    built = []

    def make(config_name, num_actors, **kw):
        built.append((config_name, num_actors, kw))
        return _GymEnv(num_actors, 17, 6)
    monkeypatch.setitem(vecenv.vecenv_config, 'B200_TEST_PLUGIN', make)
    monkeypatch.setitem(env_configurations.configurations, 'plugin_env_only_the_reference_knows', {'vecenv_type': 'B200_TEST_PLUGIN'})
    assert 'plugin_env_only_the_reference_knows' not in C.configurations
    ABI._patch(monkeypatch)
    cfg = yaml.safe_load(open(os.path.join(REF, 'rl_games', 'configs', 'mujoco', 'halfcheetah_envpool.yaml')))
    c = cfg['params']['config']
    c.update({'env_name': 'plugin_env_only_the_reference_knows', 'device': H._CudaLookingStr('cpu'), 'max_epochs': 1, 'train_dir': str(tmp_path),
              'b200_cuda_graph': False})
    runner = rl_games_b200.register(Runner())
    runner.load(cfg)
    runner.run({'train': True, 'play': False, 'checkpoint': None, 'sigma': None})
    (name, n, kw), = built
    assert name == 'plugin_env_only_the_reference_knows' and n == c['num_actors'] and kw.get('env_name') == c['env_config']['env_name']
    # a name nobody knows: the reference's own KeyError
    with pytest.raises(KeyError):
        C.create_vec_env('no_such_env_anywhere', 4)
