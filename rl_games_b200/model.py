"""Policy/value model object for the B200 PPO path.

Mirrors the call surface of the reference's ``ModelA2CContinuousLogStd.Network`` (models.py:304-364)
wrapped around ``A2CBuilder.Network`` (network_builder.py:211-593) for the subset on the hot path:
shared MLP trunk (``separate: False``), ``fixed_sigma: True`` continuous head with the 'exp' sigma
parametrisation, scalar value head, optional obs / value ``RunningMeanStd`` normalisers.

All parameters live in ONE flat fp32 arena (``self.flat``) with matching flat gradient / Adam-moment
arenas, so the optimiser, the gradient all-reduce and the checkpoint code each touch one buffer:

    [ sigma(A) | W_1 | b_1 | ... | W_L | b_L | W_head(A+1, H_L) | b_head(A+1) ]   (row 0 of the head = value)

``state_dict()`` / ``load_state_dict()`` speak the reference's key names
(``a2c_network.sigma``, ``a2c_network.actor_mlp.{0,2,..}.{weight,bias}``, ``a2c_network.value.*``,
``a2c_network.mu.*``, ``running_mean_std.*``, ``value_mean_std.*``) so checkpoints interoperate with the
reference trainer and players.
"""
import math
from collections import OrderedDict

import torch

from . import ops


def _apply_init(t, spec, fan_in):
    """network_builder.py:61-72 init_factory for the names used by shipped configs."""
    name = (spec or {}).get('name', 'default')
    kw = {k: v for k, v in (spec or {}).items() if k != 'name'}
    if name == 'default':
        bound = 1.0 / math.sqrt(fan_in)      # torch.nn.Linear default: kaiming_uniform_(a=sqrt(5))
        t.uniform_(-bound, bound)
    elif name == 'const_initializer':
        t.fill_(kw.get('val', kw.get('value', 0)))
    elif name in ('orthogonal_initializer', 'orthogonal'):
        torch.nn.init.orthogonal_(t, **kw)
    elif name == 'glorot_normal_initializer':
        torch.nn.init.xavier_normal_(t, **kw)
    elif name == 'glorot_uniform_initializer':
        torch.nn.init.xavier_uniform_(t, **kw)
    elif name == 'random_uniform_initializer':
        torch.nn.init.uniform_(t, **kw)
    elif name == 'kaiming_normal':
        torch.nn.init.kaiming_normal_(t, **kw)
    elif name == 'variance_scaling_initializer':
        # torch_ext.py:114-144 (configs/mujoco/halfcheetah*.yaml): N(0, scale / fan) by inverse CDF of uniforms drawn from NUMPY's global
        # generator (the one the runner seeds), restricted to [-2, 2] in ABSOLUTE units -- not in sigmas -- and clamped there
        import numpy as np
        sigma = math.sqrt(kw.get('scale', 2.0) / torch.nn.init._calculate_correct_fan(t, kw.get('mode', 'fan_in')))
        u = torch.from_numpy(np.random.uniform(0, 1, tuple(t.shape)))
        std_normal = torch.distributions.Normal(0.0, 1.0, validate_args=False)
        lo = std_normal.cdf(torch.tensor(-2.0 / sigma, dtype=torch.float64))
        hi = std_normal.cdf(torch.tensor(2.0 / sigma, dtype=torch.float64))
        eps = torch.finfo(torch.float64).eps
        z = (2.0 * (lo + (hi - lo) * u) - 1.0).clamp(-1.0 + eps, 1.0 - eps)
        t.copy_((sigma * math.sqrt(2.0) * torch.erfinv(z)).clamp(-2.0, 2.0))
    else:
        raise ValueError(f'unsupported initializer {name}')


class _RunningStats:
    """Device-resident RunningMeanStd state (running_mean_std.py:19-53): fp64 mean/var, int64 count,
    plus the fp32 (mean, sqrt(var+eps)) copies the fused kernels read."""

    def __init__(self, size, device):
        self.size = size
        self.running_mean = torch.zeros(size, dtype=torch.float64, device=device)
        self.running_var = torch.ones(size, dtype=torch.float64, device=device)
        self.count = torch.ones(1, dtype=torch.int64, device=device)
        self.mean_f32 = torch.zeros(size, dtype=torch.float32, device=device)
        self.std_f32 = torch.ones(size, dtype=torch.float32, device=device)
        self.refresh()

    def refresh(self):
        ops.refresh_norm(self.running_mean, self.running_var, self.mean_f32, self.std_f32)

    def state_dict(self, prefix):
        return OrderedDict([(prefix + 'running_mean', self.running_mean.clone()),
                            (prefix + 'running_var', self.running_var.clone()),
                            (prefix + 'count', self.count.reshape(()).clone())])

    def load_state_dict(self, sd, prefix=''):
        self.running_mean.copy_(sd[prefix + 'running_mean'].reshape(-1))
        self.running_var.copy_(sd[prefix + 'running_var'].reshape(-1))
        self.count.copy_(sd[prefix + 'count'].reshape(-1))
        self.refresh()

    def __call__(self, x, denorm=False):
        """Eval-mode forward (running_mean_std.py:104-113)."""
        return ops.normalize(x, self.running_mean, self.running_var, denorm=denorm)


def check_network_params(network_params):
    """Options of A2CBuilder.Network.load (network_builder.py:545-589) that change the maths and have no kernel here must fail loudly,
    never be ignored: a config that sets them would otherwise train a different network without a word."""
    name = network_params.get('name', 'actor_critic')
    if name != 'actor_critic':
        raise NotImplementedError(f"network '{name}': only 'actor_critic' (A2CBuilder) is on the B200 hot path")
    mlp = network_params['mlp']
    if mlp.get('d2rl', False):
        raise NotImplementedError('mlp.d2rl')
    if network_params.get('normalization', None) not in (None, 'None'):
        raise NotImplementedError(f"normalization: {network_params['normalization']} (layer_norm / batch_norm inside the MLP)")
    if network_params.get('joint_obs_actions', None) is not None:
        raise NotImplementedError('joint_obs_actions')
    # mlp.regularizer is read by no code path of the reference's torch builder either: ignored there, ignored here


class _NetworkView:
    """What Runner._override_sigma (torch_runner.py:52-60) touches: ``a2c_network.sigma`` / ``fixed_sigma``."""

    def __init__(self, model):
        self._m = model
        self.fixed_sigma = True

    @property
    def sigma(self):
        return self._m.sigma

    def is_rnn(self):
        return self._m.rnn_units > 0


def resolve_device(name):
    """torch.device for a config's `device` value.  An index-less 'cuda' (configs/ppo_cartpole.yaml, ppo_lunar_discrete.yaml) means the
    CURRENT device, as every torch op resolves it; it is made explicit here because raw pointers cross the C ABI and
    `torch.cuda.set_device` refuses a device without an index.  Anything else is returned as torch parses it."""
    dev = torch.device(name)
    if dev.type == 'cuda' and dev.index is None:
        dev = torch.device('cuda', torch.cuda.current_device())
    return dev


class CompileTolerantModel:
    """Mixin for agents: `Runner.run_train` of the reference wraps `agent.model` with torch.compile unless the YAML says
    `torch_compile: False` (torch_runner.py:282-312).  There is no nn.Module to compile here (the hand-written kernels subsume those
    fusions), so an assignment of anything that is not one of this package's models is ignored, once, with a note -- stock YAMLs
    run unchanged through the reference's own Runner."""

    @property
    def model(self):
        return self.__dict__.get('_b200_model')

    @model.setter
    def model(self, m):
        if self.__dict__.get('_b200_model') is not None and not hasattr(m, 'load_optimizer_state_dict'):
            if not self.__dict__.get('_b200_compile_noted'):
                print('b200: torch.compile of agent.model ignored (no nn.Module on this path; set torch_compile: False to silence)')
                self.__dict__['_b200_compile_noted'] = True
            return
        self.__dict__['_b200_model'] = m


def _model_call(self, *args, **kwargs):
    raise NotImplementedError('the B200 model is a flat parameter arena driven by fused kernels (agent.get_action_values / train_epoch); '
                              'it has no module-style forward')


def adam_opt_state(lr, step, slots=4):
    """the optimiser kernels' state row: lr, step, beta1^step, beta2^step, then zeros up to `slots`"""
    row = [float(lr), float(step), 0.9 ** float(step) if step else 0.0, 0.999 ** float(step) if step else 0.0]
    return torch.tensor(row + [0.0] * (slots - 4), dtype=torch.float64)


class FlatArena:
    """Parameters in ONE flat fp32 arena (``flat``) with matching Adam-moment arenas (``exp_avg``, ``exp_avg_sq``), so the optimiser, the
    gradient all-reduce and the checkpoint code each touch one buffer.  A subclass builds the layout from a ``(name, shape)`` list and
    defines ``_param_views(arena)``: the tensors in the reference's ``model.parameters()`` order, which the index-keyed Adam state follows.
    The generic ``state_dict`` / ``load_state_dict`` also need ``param_names()`` (the reference's keys, in the same order)."""

    def _build_arena(self, sizes, device, align=1):
        """every tensor starts on a multiple of `align` elements; the gaps hold zeros in every arena"""
        self.layout, off = OrderedDict(), 0
        for n, shp in sizes:
            off = (off + align - 1) // align * align
            self.layout[n] = (off, shp)
            off += int(torch.Size(shp).numel())
        self.num_params = off
        self.flat = torch.zeros(off, dtype=torch.float32, device=device)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)

    def _default_init(self):
        """torch.nn.Linear default weights on every W* tensor, drawn on the arena's device in layout order; biases stay zero
        (network_builder.py:332-340 with the 'default' initializer)"""
        for n, (_, shp) in self.layout.items():
            if n.startswith('W'):
                bound = 1.0 / float(shp[1]) ** 0.5
                self.view(n).uniform_(-bound, bound)

    def view(self, name, arena=None):
        off, shp = self.layout[name]
        arena = self.flat if arena is None else arena
        return arena[off:off + int(torch.Size(shp).numel())].view(shp)

    def layers(self, prefix, n):
        """[(W, b, offset of W, offset of b)] of the MLP layers W{prefix}{i} / b{prefix}{i}, i < n (see mlp_forward / mlp_backward)"""
        return [(self.view(f'W{prefix}{i}'), self.view(f'b{prefix}{i}'), self.layout[f'W{prefix}{i}'][0], self.layout[f'b{prefix}{i}'][0])
                for i in range(n)]

    def state_dict(self):
        sd = OrderedDict()
        if self.normalize_value:
            sd.update(self.value_mean_std.state_dict('value_mean_std.'))
        if self.normalize_input:
            sd.update(self.running_mean_std.state_dict('running_mean_std.'))
        for n, v in zip(self.param_names(), self._param_views(self.flat)):
            sd[n] = v.clone()
        return sd

    def load_state_dict(self, sd, strict=True):
        sd = {k.replace('_orig_mod.', ''): v for k, v in sd.items()}
        with torch.no_grad():
            for n, v in zip(self.param_names(), self._param_views(self.flat)):
                if n in sd:
                    v.copy_(sd[n].reshape(v.shape))
                elif strict:
                    raise KeyError(f'missing key in state_dict: {n}')
            self._load_normalisers(sd)

    def _load_normalisers(self, sd):
        if self.normalize_value and 'value_mean_std.running_mean' in sd:
            self.value_mean_std.load_state_dict(sd, 'value_mean_std.')
        if self.normalize_input and 'running_mean_std.running_mean' in sd:
            self.running_mean_std.load_state_dict(sd, 'running_mean_std.')

    def optimizer_state_dict(self, lr, step, weight_decay):
        """torch.optim.Adam.state_dict() layout (index-keyed, reference parameter order)."""
        state = {}
        for i, (m, v) in enumerate(zip(self._param_views(self.exp_avg), self._param_views(self.exp_avg_sq))):
            state[i] = {'step': torch.tensor(float(step)), 'exp_avg': m.clone(), 'exp_avg_sq': v.clone()}
        group = {'lr': lr, 'betas': (0.9, 0.999), 'eps': 1e-08, 'weight_decay': weight_decay, 'amsgrad': False,
                 'maximize': False, 'foreach': None, 'capturable': False, 'differentiable': False, 'fused': True,
                 'decoupled_weight_decay': False, 'params': list(range(len(state)))}
        return {'state': state, 'param_groups': [group]}

    def load_optimizer_state_dict(self, osd):
        """Returns (lr, step)."""
        st = osd.get('state', {})
        step = 0
        ms, vs = self._param_views(self.exp_avg), self._param_views(self.exp_avg_sq)
        for i in range(len(ms)):
            if i in st:
                ms[i].copy_(st[i]['exp_avg'].reshape(ms[i].shape))
                vs[i].copy_(st[i]['exp_avg_sq'].reshape(vs[i].shape))
                step = int(float(st[i]['step']))
        lr = osd['param_groups'][0]['lr'] if osd.get('param_groups') else None
        return lr, step


def mlp_forward(layers, x, acts, act_id, M, x_ld, norm, rows_per_chunk=None, chunk_stride=0, lin_fwd=None):
    """fp32 MLP trunk over M rows: layer 0 reads the observation rows of x (normalised on the fly by norm = (mean, std) or (None, None),
    optionally gathered as chunks of rows_per_chunk rows chunk_stride apart), layer i > 0 reads acts[i - 1]; activations go to acts.
    lin_fwd: the layer GEMM (default ops.linear_fwd, looked up at call time)"""
    lin_fwd = lin_fwd or ops.linear_fwd
    lin_fwd(x, layers[0][0], layers[0][1], acts[0], act_id, rows_per_chunk=rows_per_chunk, chunk_stride=chunk_stride, x_ld=x_ld,
            norm_mean=norm[0], norm_std=norm[1], M=M)
    for i in range(1, len(layers)):
        lin_fwd(acts[i - 1], layers[i][0], layers[i][1], acts[i], act_id, M=M)


def mlp_backward(layers, part, x, acts, dacts, act_id, M, x_ld, norm, rows_per_chunk, chunk_stride, lin_bwd=None, lin_bww=None):
    """Backward of mlp_forward, given dacts[-1]: the weight gradients of every layer go to the split-partial rows `part` [splits, P] at the
    layer's arena offsets, the dgrad chain fills dacts[l - 1]; layer 0's weight gradient re-reads the normalised observation rows of x.
    lin_bwd / lin_bww: the dgrad / wgrad GEMMs (default ops.linear_bwd_data / ops.linear_bwd_weight, looked up at call time)"""
    lin_bwd = lin_bwd or ops.linear_bwd_data
    lin_bww = lin_bww or ops.linear_bwd_weight
    S, P = part.shape
    for l in range(len(layers) - 1, -1, -1):
        W, _, off_w, off_b = layers[l]
        if l > 0:
            lin_bww(dacts[l], acts[l - 1], part[0, off_w:], part[0, off_b:], W.shape[1], W.shape[0], S, M=M, split_stride=P)
            lin_bwd(dacts[l], W, acts[l - 1], dacts[l - 1], act_id, M=M)
        else:
            lin_bww(dacts[0], x, part[0, off_w:], part[0, off_b:], W.shape[1], W.shape[0], S, rows_per_chunk=rows_per_chunk,
                    chunk_stride=chunk_stride, x_ld=x_ld, norm_mean=norm[0], norm_std=norm[1], M=M, split_stride=P)


class B200Model(FlatArena):
    __call__ = _model_call

    RNN_KEYS = (('a2c_network.rnn.rnn.weight_ih_l0', 'W_ih'), ('a2c_network.rnn.rnn.weight_hh_l0', 'W_hh'),
                ('a2c_network.rnn.rnn.bias_ih_l0', 'b_ih'), ('a2c_network.rnn.rnn.bias_hh_l0', 'b_hh'))

    def __init__(self, network_params, obs_dim, act_dim, device, normalize_input, normalize_value, value_size=1,
                 seed=None):
        if value_size != 1:
            raise NotImplementedError('value_size > 1 is not on the B200 hot path yet')
        check_network_params(network_params)
        mlp = network_params['mlp']
        self.units = list(mlp['units'])
        if len(self.units) == 0:
            raise NotImplementedError('empty MLP')
        self.activation = mlp.get('activation', 'elu')
        if self.activation not in ops.ACT:
            raise NotImplementedError(f'activation {self.activation}')
        self.act_id = ops.ACT[self.activation]
        # separate: True (network_builder.py:494-512; configs/ppo_continuous.yaml, ppo_lunar.yaml ...): actor_mlp feeds mu, critic_mlp feeds the
        # value.  Here the two trunks are ONE MLP of twice the width whose weights are block-structured -- layer 0 stacks [W_actor; W_critic] (both
        # read the observation), layers >= 1 are block-diagonal, the value row of the head reads the critic half and the mu rows the actor half --
        # so every kernel, arena and code path of the shared-trunk policy is used as it is.  The structural zeros stay exactly zero: their
        # gradient entries are masked before the optimiser (grad_mask), and a zero weight with a zero gradient is a fixed point of Adam and of
        # weight decay; multiplied by zero they add exact zeros to the products.  `units` = the EFFECTIVE widths everything downstream sees,
        # `trunk_units` = the reference's per-trunk widths (state-dict shapes).
        self.separate = bool(network_params.get('separate', False))
        self.trunk_units = list(self.units)
        if self.separate:
            if 'rnn' in network_params:
                raise NotImplementedError('separate actor/critic trunks with an rnn (two recurrent cores) are not on the B200 hot path')
            self.units = [2 * u for u in self.trunk_units]
        if 'cnn' in network_params:
            raise NotImplementedError("'cnn' networks are not on the B200 hot path yet")
        self.rnn_units = 0
        if 'rnn' in network_params:
            rnn = network_params['rnn']
            if rnn.get('name') != 'lstm' or rnn.get('layers', 1) != 1 or rnn.get('layer_norm', False) \
                    or rnn.get('concat_input', False) or rnn.get('concat_output', False):
                raise NotImplementedError("rnn: only a single-layer 'lstm' (no layer_norm / concat) is on the B200 hot path")
            self.rnn_units = int(rnn['units'])
        # placement (network_builder.py:253-272): before_mlp True = obs -> LSTM -> MLP -> heads (BASELINE configs[3]); False (the reference
        # default) = obs -> MLP -> LSTM -> heads.  Same parameter names and order either way, different shapes.
        self.rnn_before_mlp = bool(network_params.get('rnn', {}).get('before_mlp', False)) if self.rnn_units else True
        space = network_params['space']['continuous']
        if not space.get('fixed_sigma', True):
            raise NotImplementedError('state-dependent sigma is not on the B200 hot path yet')
        for k in ('mu_activation', 'sigma_activation'):
            if space.get(k, 'None') not in ('None', None):
                raise NotImplementedError(f'{k}={space[k]}')
        if space.get('sigma_parametrization', 'exp') != 'exp' or space.get('logstd_bounds'):
            raise NotImplementedError("only the 'exp' sigma parametrisation (optionally floored by min_sigma) is on the B200 hot path")
        # models.py:272-300, 'exp' branch with a floor (configs/mjlab/ppo_lift_cube_yam.yaml: min_sigma 0.15): sigma = exp(raw) + min_sigma
        self.min_sigma = float(space.get('min_sigma', 0.0) or 0.0)
        if network_params.get('value_activation', 'None') not in ('None', None):
            raise NotImplementedError('value_activation')
        self.D, self.A = int(obs_dim), int(act_dim)
        self.device = torch.device(device)
        self.normalize_input, self.normalize_value = bool(normalize_input), bool(normalize_value)
        # ---- flat arenas ----
        sizes = [('sigma', (self.A,))]
        Hd = self.rnn_units
        self.rnn_in = (self.D if self.rnn_before_mlp else self.units[-1]) if Hd else 0      # input width of the LSTM
        if Hd:
            sizes += [('W_ih', (4 * Hd, self.rnn_in)), ('W_hh', (4 * Hd, Hd)), ('b_ih', (4 * Hd,)), ('b_hh', (4 * Hd,))]
        ins = Hd if (Hd and self.rnn_before_mlp) else self.D
        for i, u in enumerate(self.units):
            sizes += [(f'W{i}', (u, ins)), (f'b{i}', (u,))]
            ins = u
        if Hd and not self.rnn_before_mlp:
            ins = Hd                     # the heads read the LSTM output
        self.Hl = ins
        sizes += [('W_head', (self.A + 1, ins)), ('b_head', (self.A + 1,))]
        # every tensor starts on an 8-element boundary (32 bytes in the fp32 arenas, 16 bytes in the bf16 twin the tensor-core GEMMs
        # read): weight rows can then be staged with 16-byte loads whatever the action count did to the offsets.  The gaps hold
        # zeros in every arena (weights, gradients, moments), so norms, Adam and the all-reduce are unaffected; layouts whose tensor
        # sizes are all multiples of 8 (the BASELINE MLPs with 8 actions) have no gaps at all.
        self._build_arena(sizes, self.device, align=8)
        off = self.num_params
        self.grad = torch.zeros(off, dtype=torch.float32, device=self.device)
        self.W =[self.view(f'W{i}') for i in range(len(self.units))]
        self.b = [self.view(f'b{i}') for i in range(len(self.units))]
        self.sigma = self.view('sigma')
        if self.min_sigma > 0:
            # what the kernels are handed instead of the raw parameter, and the chain factor of its gradient (refresh_sigma_floor)
            self.logstd_eff = torch.zeros(self.A, dtype=torch.float32, device=self.device)
            self.sigma_chain = torch.ones(self.A, dtype=torch.float32, device=self.device)
        if self.rnn_units:
            self.W_ih, self.W_hh, self.b_ih, self.b_hh = (self.view(n) for n in ('W_ih', 'W_hh', 'b_ih', 'b_hh'))
        self.mlp_in = self.rnn_units if (self.rnn_units and self.rnn_before_mlp) else self.D
        self.W_head, self.b_head = self.view('W_head'), self.view('b_head')
        self.grad_mask = None
        if self.separate:       # 1 on the entries the reference has a parameter for, 0 on the structural zeros of the block layout
            self.grad_mask = torch.zeros(off, dtype=torch.float32, device=self.device)
            for v in self._param_views(self.grad_mask):
                v.fill_(1.0)
        self.gW = [self.view(f'W{i}', self.grad) for i in range(len(self.units))]
        self.gb = [self.view(f'b{i}', self.grad) for i in range(len(self.units))]
        self.g_sigma = self.view('sigma', self.grad)
        self.gW_head, self.gb_head = self.view('W_head', self.grad), self.view('b_head', self.grad)
        self.running_mean_std = _RunningStats(self.D, self.device) if self.normalize_input else None
        self.value_mean_std = _RunningStats(1, self.device)   # always allocated; used iff normalize_value
        self.a2c_network = _NetworkView(self)
        self._init_weights(network_params, seed)
        self.training = False

    # -------------------------------------------------------------------------------------------
    @property
    def logstd_in(self):
        """The log-std vector the policy kernels read.  They compute sigma = exp(logstd) -- with a floor (min_sigma > 0) that is the
        EFFECTIVE log-std log(exp(raw) + min_sigma) (models.py:296-300: `sigma + min_sigma`, `logstd = log(sigma)`), kept in its own
        buffer by refresh_sigma_floor(); without a floor it is the parameter itself."""
        return self.logstd_eff if self.min_sigma > 0 else self.sigma

    def refresh_sigma_floor(self):
        """After anything that changes the raw sigma parameter (optimiser step, weight load): logstd_eff = log(e^raw + min_sigma) and
        sigma_chain = d logstd_eff / d raw = e^raw / (e^raw + min_sigma), the factor that turns the kernels' gradient with respect to
        the log-std they were handed into the gradient of the raw parameter.  Three in-place launches on [A] vectors, no allocation
        (CUDA-graph capturable); a no-op without a floor."""
        if self.min_sigma > 0:
            torch.exp(self.sigma, out=self.sigma_chain)
            torch.add(self.sigma_chain, self.min_sigma, out=self.logstd_eff)
            self.sigma_chain.div_(self.logstd_eff)
            self.logstd_eff.log_()

    def _init_weights(self, network_params, seed):
        """network_builder.py:326-348: mlp initializer on every Linear weight, zero biases, mu_init on mu.weight,
        sigma_init on the sigma parameter."""
        space = network_params['space']['continuous']
        mlp_init = network_params['mlp'].get('initializer', {'name': 'default'})
        cpu = {}
        if self.rnn_units:   # torch.nn.LSTM default init U(-1/sqrt(hid), 1/sqrt(hid)) for all four tensors (mlp_init does not touch it)
            Hd = self.rnn_units
            k = 1.0 / math.sqrt(Hd)
            for n, shp in (('W_ih', (4 * Hd, self.rnn_in)), ('W_hh', (4 * Hd, Hd)), ('b_ih', (4 * Hd,)), ('b_hh', (4 * Hd,))):
                cpu[n] = torch.empty(*shp).uniform_(-k, k)
        mu_init = space.get('mu_init', {'name': 'default'})
        if self.separate:       # every Linear of both trunks and both heads is initialised on its own (true fan-in), written into its block
            blocks = self._param_views(self.flat)[1:]               # actor W, b ... critic W, b ... value W, b, mu W, b
            for k in range(0, len(blocks), 2):
                w = torch.empty(*blocks[k].shape)
                _apply_init(w, mlp_init, w.shape[1])
                if k == len(blocks) - 2 and mu_init.get('name', 'default') != 'default':
                    _apply_init(w, mu_init, w.shape[1])
                blocks[k].copy_(w)
        else:
            ins = self.mlp_in
            for i, u in enumerate(self.units):
                w = torch.empty(u, ins)
                _apply_init(w, mlp_init, ins)
                cpu[f'W{i}'] = w
                ins = u
            ins = self.Hl
            wh = torch.empty(self.A + 1, ins)
            _apply_init(wh[:1], mlp_init, ins)                                   # value head: mlp_init
            _apply_init(wh[1:], mlp_init, ins)
            if mu_init.get('name', 'default') != 'default':
                _apply_init(wh[1:], mu_init, ins)
            cpu['W_head'] = wh
        sg = torch.empty(self.A)
        _apply_init(sg, space.get('sigma_init', {'name': 'const_initializer', 'val': 0}), 1)
        cpu['sigma'] = sg
        for n, t in cpu.items():
            self.view(n).copy_(t)

    # ------------------------------------------------------------------------------------------- nn.Module-ish
    def is_rnn(self):
        return self.rnn_units > 0

    def get_default_rnn_state(self, num_seqs=1):
        """network_builder.py:520-543 (lstm, not separate): (h, c) each [layers, num_seqs, units]"""
        if not self.rnn_units:
            return None
        return (torch.zeros((1, num_seqs, self.rnn_units), device=self.device), torch.zeros((1, num_seqs, self.rnn_units), device=self.device))

    def get_aux_loss(self):
        return None

    def eval(self):
        self.training = False
        return self

    def train(self, mode=True):
        self.training = mode
        return self

    def to(self, device):
        return self

    def parameters(self):
        """Reference parameter order (optimizer state is index-keyed): sigma, actor_mlp.*, value.*, mu.*"""
        return self._param_views(self.flat)

    def _param_views(self, arena):
        if self.separate:
            return self._param_views_separate(arena)
        out = [self.view('sigma', arena)]
        for i in range(len(self.units)):
            out += [self.view(f'W{i}', arena), self.view(f'b{i}', arena)]
        if self.rnn_units:   # registration order in A2CBuilder.Network.__init__: actor_mlp placeholder precedes self.rnn
            out += [self.view(n, arena) for n in ('W_ih', 'W_hh', 'b_ih', 'b_hh')]
        wh, bh = self.view('W_head', arena), self.view('b_head', arena)
        out += [wh[:1], bh[:1], wh[1:], bh[1:]]
        return out

    def _param_views_separate(self, arena):
        """separate: True -- the reference's parameters (order: sigma, actor_mlp.*, critic_mlp.*, value.*, mu.*) as block views of the
        double-width layout: trunk t of layer i owns rows [t u_i, (t + 1) u_i); layer 0 reads all observation columns, layers >= 1 the
        columns [t u_(i-1), (t + 1) u_(i-1)) of their own trunk; value = head row 0 on the critic half, mu = head rows 1.. on the actor half"""
        tu = self.trunk_units
        out = [self.view('sigma', arena)]
        for t in (0, 1):
            for i, u in enumerate(tu):
                w, b = self.view(f'W{i}', arena), self.view(f'b{i}', arena)
                cols = slice(None) if i == 0 else slice(t * tu[i - 1], (t + 1) * tu[i - 1])
                out += [w[t * u:(t + 1) * u, cols], b[t * u:(t + 1) * u]]
        wh, bh = self.view('W_head', arena), self.view('b_head', arena)
        out += [wh[:1, tu[-1]:], bh[:1], wh[1:, :tu[-1]], bh[1:]]
        return out

    def _separate_keys(self):
        keys = ['a2c_network.sigma']
        for trunk in ('actor_mlp', 'critic_mlp'):
            for i in range(len(self.trunk_units)):
                keys += [f'a2c_network.{trunk}.{2 * i}.weight', f'a2c_network.{trunk}.{2 * i}.bias']
        return keys + ['a2c_network.value.weight', 'a2c_network.value.bias', 'a2c_network.mu.weight', 'a2c_network.mu.bias']

    def state_dict(self):
        sd = OrderedDict()
        if self.normalize_value:
            sd.update(self.value_mean_std.state_dict('value_mean_std.'))
        if self.normalize_input:
            sd.update(self.running_mean_std.state_dict('running_mean_std.'))
        if self.separate:
            for k, v in zip(self._separate_keys(), self._param_views(self.flat)):
                sd[k] = v.clone()
            return sd
        sd['a2c_network.sigma'] = self.sigma.clone()
        for i in range(len(self.units)):
            sd[f'a2c_network.actor_mlp.{2 * i}.weight'] = self.W[i].clone()
            sd[f'a2c_network.actor_mlp.{2 * i}.bias'] = self.b[i].clone()
        for key, n in self.RNN_KEYS:
            if self.rnn_units:
                sd[key] = self.view(n).clone()
        sd['a2c_network.value.weight'] = self.W_head[:1].clone()
        sd['a2c_network.value.bias'] = self.b_head[:1].clone()
        sd['a2c_network.mu.weight'] = self.W_head[1:].clone()
        sd['a2c_network.mu.bias'] = self.b_head[1:].clone()
        return sd

    def load_state_dict(self, sd, strict=True):
        sd = {k.replace('_orig_mod.', ''): v for k, v in sd.items()}
        need = [k for k in self.state_dict().keys()]
        missing = [k for k in need if k not in sd]
        if missing and strict:
            raise KeyError(f'missing keys in state_dict: {missing}')
        with torch.no_grad():
            if self.separate:
                for k, v in zip(self._separate_keys(), self._param_views(self.flat)):
                    if k in sd:
                        v.copy_(sd[k].reshape(v.shape))
                self._load_normalisers(sd)
                return
            if 'a2c_network.sigma' in sd:
                self.sigma.copy_(sd['a2c_network.sigma'])
            for i in range(len(self.units)):
                self.W[i].copy_(sd[f'a2c_network.actor_mlp.{2 * i}.weight'])
                self.b[i].copy_(sd[f'a2c_network.actor_mlp.{2 * i}.bias'])
            if self.rnn_units:
                for key, n in self.RNN_KEYS:
                    self.view(n).copy_(sd[key])
            self.W_head[:1].copy_(sd['a2c_network.value.weight'])
            self.b_head[:1].copy_(sd['a2c_network.value.bias'])
            self.W_head[1:].copy_(sd['a2c_network.mu.weight'])
            self.b_head[1:].copy_(sd['a2c_network.mu.bias'])
            self._load_normalisers(sd)

