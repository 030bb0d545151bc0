"""Central value (asymmetric critic) on top of the continuous B200 agent -- SURVEY.md 8f rank 1 (reference:
algos_torch/central_value.py CentralValueTrain, models.py:425-464 ModelCentralValue, a2c_common.py:250-262, :593-615, :1010-1011,
:1536-1537, :1651-1660; a2c_continuous.py:50-75).

STATUS: parity-green on a B200 (round 2, ``tests/test_cv_gpu.py``).  The reference
semantics are pinned by ``oracle.ppo_oracle.CentralValueOracle`` against ``tests/golden/agent_cv.pt``; the HOST logic of this module runs
on CPU against the same golden vectors with torch stand-ins for the kernels (``tests/test_agent_cv_host_cpu.py``); the only new kernel
(``csrc/critic.cu`` value loss) has its row arithmetic exercised on the CPU too.  Everything else reuses validated kernels.

``A2CAgentCV`` subclasses the validated ``A2CAgent`` without touching it:
  * the env returns ``{'obs': actor view, 'states': privileged critic view}``; ``states`` go to the critic's arena;
  * rollout values / the last value come from the critic (de-normalised with ITS value normaliser), so the time-out bootstrap and
    GAE use them; the agent's value normaliser IS the critic's (a2c_continuous.py:72-73);
  * the critic trains (own minibatching, own Adam, own obs normaliser re-armed on every minibatch) before the actor's mini-epochs;
  * the actor keeps its own value head and value loss (``use_experimental_cv`` defaults to True in the reference).
Precision is the critic's own key, ``central_value_config['mixed_precision']`` (central_value.py:24), never the agent's:
  * True: every trunk layer runs on the layer-wise tcgen05 GEMMs (``gemm_tc.cu``: bf16 operands from a bf16 twin of the critic's arena,
    fp32 accumulate), in training and in the rollout; the 1-wide value head is one fused fp32 kernel (``csrc/critic.cu``
    value_head_loss / value_head_fwd).  Rollout and last values come from the same kernels as training, so old and re-evaluated values
    share arithmetic (DESIGN.md §2, §8).  The twin is refreshed after every critic optimiser step and every weight load;
  * False: the fp32 CUDA-core kernels;
  * absent: the fp32 kernels, with a printed note.
``central_value_net.gemm_tc`` records the result.  The tensor-core critic's host logic is checked on CPU (``tests/test_cv_tensor_cores_cpu.py``);
its GPU tests (``tests/test_cv_tensor_cores_gpu.py``) have not yet run on hardware.
Scope: MLP critic, no whole-epoch CUDA graph (the update-phase graph of the actor still works), identity / linear critic LR schedule.
"""
from collections import OrderedDict

import torch
import torch.distributed as dist

from . import ops
from .agent import A2CAgent
from .common import IdentityScheduler, LinearScheduler
from .model import _RunningStats, FlatArena, adam_opt_state, check_network_params, mlp_backward, mlp_forward


class CentralValueNet(FlatArena):
    """CentralValueTrain on the fp32 kernels: flat arena [W0 b0 ... W_v b_v] in the reference's parameter order."""

    # `CentralValueTrain.model` (central_value.py:44): the reference's Runner wraps it with torch.compile unless the YAML says
    # `torch_compile: False` (torch_runner.py:308-313).  Here the net IS its model and there is no nn.Module to compile: reading `.model`
    # gives the net, assigning anything else to it is ignored with a note (like CompileTolerantModel does for `agent.model`).
    @property
    def model(self):
        return self

    @model.setter
    def model(self, m):
        if m is not self and not self.__dict__.get('_b200_compile_noted'):
            print('b200: torch.compile of central_value_net.model ignored (no nn.Module on this path; set torch_compile: False to silence)')
            self.__dict__['_b200_compile_noted'] = True

    def __call__(self, *args, **kwargs):
        raise NotImplementedError('the central value net is a flat parameter arena driven by kernels (get_value / train_net); '
                                  'it has no module-style forward')

    def __init__(self, cv_config, state_dim, num_actors, horizon, normalize_value, max_epochs, device, multi_gpu=False, world_size=1):
        net = cv_config['network']
        self.multi_gpu, self.world_size = bool(multi_gpu) and world_size > 1, int(world_size)
        self.writter = None             # the agent's summary writer (central_value.py:79; the reference's spelling)
        check_network_params(net)
        mlp = net['mlp']
        self.units = list(mlp['units'])
        self.activation = mlp.get('activation', 'elu')
        if self.activation not in ops.ACT or not self.units or any(k in net for k in ('cnn', 'rnn')):
            raise NotImplementedError('central value network: a plain MLP is supported')
        self.act_id = ops.ACT[self.activation]
        self.S, self.N, self.H = int(state_dim), int(num_actors), int(horizon)
        self.device = torch.device(device)
        self.normalize_input, self.normalize_value = bool(cv_config['normalize_input']), bool(normalize_value)
        self.lr = float(cv_config['learning_rate'])
        self.mini_epoch = int(cv_config['mini_epochs'])
        self.batch_size = self.N * self.H
        if 'minibatch_size' not in cv_config and 'minibatch_size_per_env' not in cv_config:
            raise ValueError("Configuration must include either 'minibatch_size' or 'minibatch_size_per_env'. "
                             "Neither was found in the provided config.")
        self.minibatch_size = int(cv_config.get('minibatch_size', self.N * cv_config.get('minibatch_size_per_env', 0)))
        if self.minibatch_size <= 0 or self.batch_size % self.minibatch_size or self.minibatch_size % self.H:
            raise NotImplementedError('central value minibatch_size must divide the batch and be a multiple of horizon_length')
        self.num_minibatches = self.batch_size // self.minibatch_size
        self.envs_per_mb = self.minibatch_size // self.H
        self.clip_value, self.e_clip = bool(cv_config['clip_value']), float(cv_config.get('e_clip', 0.2))
        self.truncate_grads, self.grad_norm = bool(cv_config.get('truncate_grads', False)), float(cv_config.get('grad_norm', 1))
        self.weight_decay = float(cv_config.get('weight_decay', 0.0))
        self.freeze = bool(cv_config.get('freeze_critic', False))
        # precision (central_value.py:24): the critic's own key, never the agent's.  True -> trunk on the layer-wise tcgen05 GEMMs
        # (bf16 operands, fp32 accumulate) and the fused fp32 value head; False or absent -> the fp32 CUDA-core kernels
        self.precision_set = 'mixed_precision' in cv_config
        self.gemm_tc = bool(cv_config.get('mixed_precision', False))
        self.scheduler = (LinearScheduler(self.lr, max_steps=max_epochs, apply_to_entropy=False, start_entropy_coef=0)
                          if cv_config.get('lr_schedule') == 'linear' else IdentityScheduler())        # central_value.py:55-62
        self.epoch_num = self.frame = 0
        sizes, ins = [], self.S
        for i, u in enumerate(self.units):
            sizes += [(f'W{i}', (u, ins)), (f'b{i}', (u,))]
            ins = u
        self.Hl = ins
        if self.gemm_tc and self.Hl > ops.VALUE_HEAD_MAX_HL:
            raise NotImplementedError(f'central value mixed_precision: the fused value head takes a last layer of at most '
                                      f'{ops.VALUE_HEAD_MAX_HL} units (got {self.Hl})')
        sizes += [('W_v', (1, ins)), ('b_v', (1,))]
        dev = self.device
        self._build_arena(sizes, dev)
        off = self.num_params
        self._default_init()
        self.running_mean_std = _RunningStats(self.S, dev) if self.normalize_input else None
        self.value_mean_std = _RunningStats(1, dev) if self.normalize_value else None
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)   # noqa: E731
        mb = self.minibatch_size
        self.states = f(self.H, self.N, self.S)
        self.r_act = [f(self.N, u) for u in self.units]
        self.t_act = [f(mb, u) for u in self.units]
        self.d_act = [f(mb, u) for u in self.units]
        self.r_val, self.t_val, self.d_val = f(self.N, 1), f(mb, 1), f(mb, 1)
        # split rows of the weight gradients: the tensor-core GEMMs are sized like the actor's layer-wise path (agent.py)
        self.n_splits = max(1, min(16, mb // 512)) if self.gemm_tc else max(1, min(64, mb // 256))
        self.part = f(self.n_splits, off)
        self.grad = f(off)
        self.loss_partials = torch.zeros((mb + 255) // 256, 8, dtype=torch.float64, device=dev)
        self.inv_counts = f(self.num_minibatches)
        self.mom_scratch = torch.zeros(148 * 4 * 2 * self.S, dtype=torch.float64, device=dev)
        self.counters = torch.zeros(4, dtype=torch.int32, device=dev)
        self.opt_state = adam_opt_state(self.lr, 0).to(dev)
        self.adam_stats = f(16)
        # grad_scale = 1/world: the optimiser kernel scales the SUM the all-reduce leaves in self.grad (central_value.py:322-337)
        self.opt_cfg = ops.OptCfg(0.9, 0.999, 1e-8, self.weight_decay, self.grad_norm, 0.0, 1e-6, 1e-2, 1.5,
                                  1.0 / (self.world_size if self.multi_gpu else 1), int(self.truncate_grads), 0)
        self.last_losses = []
        if self.gemm_tc:
            self.wbf = torch.empty(off, dtype=torch.bfloat16, device=dev)      # bf16 twin of the arena: the GEMMs' weight operands
            self.refresh_twin()

    def param_names(self):
        names = []
        for i in range(len(self.units)):
            names += [f'a2c_network.actor_mlp.{2 * i}.weight', f'a2c_network.actor_mlp.{2 * i}.bias']
        return names + ['a2c_network.value.weight', 'a2c_network.value.bias']

    def _param_views(self, arena=None):
        out = []
        for i in range(len(self.units)):
            out += [self.view(f'W{i}', arena), self.view(f'b{i}', arena)]
        return out + [self.view('W_v', arena), self.view('b_v', arena)]

    def load_state_dict(self, sd, strict=True):
        def strip(k):          # CentralValueTrain.state_dict() prefixes its model's keys with 'model.'; torch.compile adds '_orig_mod.'
            k = k.replace('_orig_mod.', '')
            return k[len('model.'):] if k.startswith('model.') else k
        super().load_state_dict({strip(k): v for k, v in sd.items()}, strict)
        self.refresh_twin()

    def refresh_twin(self):
        """the tensor-core GEMMs read the bf16 twin of the arena: refreshed after every optimiser step and every weight load (a stale
        twin gives plausible values from the old weights)"""
        if self.gemm_tc:
            ops.cast_bf16(self.flat, self.wbf)

    # layer GEMMs of the selected precision (looked up at call time: the ops may be replaced after construction)
    def _lin_fwd(self, *a, **k):
        if self.gemm_tc:
            ops.linear_fwd_tc(*a, bf16_arena=(self.flat, self.wbf), **k)
        else:
            ops.linear_fwd(*a, **k)

    def _lin_bwd(self, *a, **k):
        if self.gemm_tc:
            ops.linear_bwd_data_tc(*a, bf16_arena=(self.flat, self.wbf), **k)
        else:
            ops.linear_bwd_data(*a, **k)

    def _lin_bww(self, *a, **k):
        (ops.linear_bwd_weight_tc if self.gemm_tc else ops.linear_bwd_weight)(*a, **k)

    # ---------------------------------------------------------------------------------------------- forward
    def _norm(self):
        r = self.running_mean_std
        return (r.mean_f32, r.std_f32) if self.normalize_input else (None, None)

    def _trunk(self, x, acts, M, rows_per_chunk=None, chunk_stride=0):
        mlp_forward(self.layers('', len(self.units)), x, acts, self.act_id, M, self.S, self._norm(), rows_per_chunk, chunk_stride,
                    lin_fwd=self._lin_fwd)

    def get_value(self, states, out):
        """central_value.py:207-229 (eval mode): out[N] = denorm(critic(states))"""
        self._trunk(states, self.r_act, self.N)
        if self.gemm_tc:        # the fused head: same GEMV arithmetic as training's, de-normalisation in the same launch
            vm = self.value_mean_std if self.normalize_value else None
            ops.value_head_fwd(self.r_act[-1], self.view('W_v'), self.view('b_v'), None if vm is None else vm.running_mean,
                               None if vm is None else vm.running_var, self.normalize_value, out, self.N)
            return
        ops.linear_fwd(self.r_act[-1], self.view('W_v'), self.view('b_v'), self.r_val, 0, M=self.N)
        if self.normalize_value:
            vm = self.value_mean_std
            ops.normalize(self.r_val, vm.running_mean, vm.running_var, denorm=True, out=out.view(self.N, 1))
        else:
            out.copy_(self.r_val.view(-1))

    # ---------------------------------------------------------------------------------------------- training (central_value.py:246-274)
    def train_net(self, old_values_n, returns_n, valid):
        H, N, mb, epm, P, S_ = self.H, self.N, self.minibatch_size, self.envs_per_mb, self.num_params, self.n_splits
        if valid is not None:
            ops.mask_inv_counts(valid, H, N, epm, self.inv_counts)
        rows = []
        for _ in range(self.mini_epoch):
            if self.freeze:
                break
            for i in range(self.num_minibatches):
                e0 = i * epm
                x = self.states[0, e0:]
                if self.normalize_input:      # train_critic -> self.train() re-arms the critic's obs normaliser on every minibatch
                    r = self.running_mean_std
                    ops.moments_update(x, self.S, epm, H, N, r.running_mean, r.running_var, r.count, r.mean_f32, r.std_f32, self.mom_scratch,
                                       self.counters[1:2])
                self._trunk(x, self.t_act, mb, rows_per_chunk=epm, chunk_stride=N)
                off_w, _ = self.layout['W_v']
                off_b, _ = self.layout['b_v']
                mask, inv = (None, None) if valid is None else (valid[0, e0:], self.inv_counts[i:i + 1])
                if self.gemm_tc:        # value GEMV + loss + d(a_last) + head gradient in one launch
                    nb = ops.value_head_loss(self.t_act[-1], self.view('W_v'), self.view('b_v'), old_values_n[0, e0:], returns_n[0, e0:], mask,
                                             epm, N, mb, self.e_clip, self.clip_value, inv, self.act_id, self.d_act[-1], self.part[0, off_w:],
                                             self.part[0, off_b:], P, S_, self.loss_partials)
                    rows.append(self.loss_partials[:nb, 0].sum().float())
                else:
                    ops.linear_fwd(self.t_act[-1], self.view('W_v'), self.view('b_v'), self.t_val, 0, M=mb)
                    nb = ops.value_loss(self.t_val, 1, old_values_n[0, e0:], returns_n[0, e0:], mask, epm, N, mb, self.e_clip, self.clip_value,
                                        inv, self.d_val, 1, self.loss_partials)
                    rows.append(self.loss_partials[:nb, 0].sum().float())
                    ops.linear_bwd_weight(self.d_val, self.t_act[-1], self.part[0, off_w:], self.part[0, off_b:], self.Hl, 1, S_, M=mb,
                                          split_stride=P)
                    ops.linear_bwd_data(self.d_val, self.view('W_v'), self.t_act[-1], self.d_act[-1], self.act_id, M=mb)
                mlp_backward(self.layers('', len(self.units)), self.part, x, self.t_act, self.d_act, self.act_id, mb, self.S, self._norm(),
                             epm, N, lin_bwd=self._lin_bwd, lin_bww=self._lin_bww)
                ops.reduce_splits(self.part, self.grad, P, S_, split_stride=P)
                if self.multi_gpu:      # the critic's own flat-gradient exchange, one per minibatch (central_value.py:322-337)
                    dist.all_reduce(self.grad, op=dist.ReduceOp.SUM)
                ops.adam_step(self.flat, self.grad, self.exp_avg, self.exp_avg_sq, self.opt_state, None, self.opt_cfg, self.adam_stats,
                              self.counters[2:3], n=P)
                self.refresh_twin()         # on every rank, after the exchange: the next minibatch's GEMMs read the new weights
        self.last_losses = rows
        self.epoch_num += 1
        self.lr, _ = self.scheduler.update(self.lr, 0, self.epoch_num, self.frame, 0)
        self.opt_state[0] = self.lr
        self.frame += self.batch_size
        if self.writter is not None and rows:       # central_value.py:262-272 (one read-back per epoch, like the reference's add_scalar)
            self.writter.add_scalar('losses/cval_loss', float(torch.stack(rows).sum()) / (self.mini_epoch * self.num_minibatches), self.frame)
            self.writter.add_scalar('info/cval_lr', self.lr, self.frame)
        return rows


class A2CAgentCV(A2CAgent):
    def __init__(self, base_name, params):
        config = params['config']
        cv_config = config.get('central_value_config')
        if cv_config is None:
            raise ValueError('A2CAgentCV needs central_value_config')
        config['central_value_config'] = None          # the base class refuses it; everything it builds is unchanged by the critic
        try:
            super().__init__(base_name, params)
        finally:
            config['central_value_config'] = cv_config
        self.central_value_config = cv_config
        self.has_central_value = True
        self.use_experimental_cv = config.get('use_experimental_cv', True)
        if not self.use_experimental_cv:
            raise NotImplementedError('use_experimental_cv: False (actor without a value loss)')
        space = self.env_info.get('state_space', None) or self.observation_space           # a2c_common.py:254-262
        if type(space).__name__ == 'Dict' or len(space.shape) != 1:
            raise NotImplementedError('only flat state spaces')
        self.state_shape = space.shape
        self.central_value_net = CentralValueNet(cv_config, space.shape[0], self.num_actors, self.horizon_length, self.normalize_value,
                                                 self.max_epochs, self.device_t, multi_gpu=self.multi_gpu, world_size=self.world_size)
        self.central_value_net.writter = self.writer
        self.value_mean_std = self.central_value_net.value_mean_std                        # a2c_continuous.py:72-73
        if not self.central_value_net.precision_set and self.global_rank == 0:
            print('b200: central_value_config.mixed_precision not set -> fp32 kernels for the critic; mixed_precision: True in '
                  'central_value_config runs its layers on the tensor cores (bf16 operands, fp32 accumulate)')
        self._states = None

    # ---- env plumbing: keep the privileged view
    def obs_to_tensors(self, obs):
        if isinstance(obs, dict) and 'states' in obs:
            self._states = self.cast_obs(obs['states'], name='states')
        elif not isinstance(obs, dict) and self.env_info.get('state_space', None) is None:
            self._states = self.cast_obs(obs, name='states')          # state_space fallback = observation_space
        return super().obs_to_tensors(obs)

    # ---- rollout: the critic supplies the values (a2c_common.py:593-600, :603-615, :1010-1011)
    def _policy_step(self, obs, t, noise=None):
        super()._policy_step(obs, t, noise)
        cv = self.central_value_net
        cv.states[t].copy_(self._states)
        cv.get_value(self._states, self.values[t])

    def get_values(self, obs):
        self.central_value_net.get_value(self._states, self.last_values)

    def _whole_epoch_graph_ok(self):
        return False                                   # the critic's training is eager

    def _stats_modules(self):
        """a2c_common.py:753-765: the cross-rank running-stat sync also covers the critic's normalisers (the value normaliser the
        agent uses IS the critic's; the actor model's own never moves and merges as a no-op delta)"""
        mods = super()._stats_modules()
        cv = self.central_value_net
        if cv.running_mean_std is not None:
            mods.append(('cv_obs', cv.running_mean_std))
        if cv.value_mean_std is not None:
            mods.append(('cv_value', cv.value_mean_std))
        return mods

    # ---- the agent's value normaliser is the critic's
    def _prepare(self, n_partials):
        m, keep = self.model, self.model.value_mean_std
        m.value_mean_std = self.central_value_net.value_mean_std
        try:
            super()._prepare(n_partials)
        finally:
            m.value_mean_std = keep

    # ---- the critic trains before the actor's mini-epochs (a2c_common.py:1536-1537)
    def _run_update(self):
        self.central_value_net.train_net(self.old_values_n, self.returns_n, self.valid)
        super()._run_update()

    def train_central_value(self):
        return self.central_value_net.train_net(self.old_values_n, self.returns_n, self.valid)

    # ---- checkpoints (a2c_common.py:831-833, :859-862)
    def get_full_state_weights(self):
        state = super().get_full_state_weights()
        cv = self.central_value_net
        state['assymetric_vf_nets'] = OrderedDict(('model.' + k, v) for k, v in cv.state_dict().items())
        st = {i: {'step': torch.tensor(float(cv.opt_state.cpu()[1])), 'exp_avg': m.clone(), 'exp_avg_sq': v.clone()}
              for i, (m, v) in enumerate(zip(cv._param_views(cv.exp_avg), cv._param_views(cv.exp_avg_sq)))}
        state['assymetric_vf_optimizer'] = {'state': st, 'param_groups': [{'lr': cv.lr, 'betas': (0.9, 0.999), 'eps': 1e-08,
                                                                          'weight_decay': cv.weight_decay, 'params': list(range(len(st)))}]}
        return state

    def restore_central_value_function(self, fn):
        """a2c_continuous.py:90-92: the critic's weights and normalisers only (`load_critic_only` of the Runner, torch_runner.py:43-50)"""
        checkpoint = torch.load(fn, map_location=self.device_t, weights_only=False)
        self.set_central_value_function_weights(checkpoint)

    def set_central_value_function_weights(self, weights):
        """a2c_common.py:885-887"""
        self.central_value_net.load_state_dict(weights['assymetric_vf_nets'])
        self._seed_stats_sync_snapshots()

    def set_full_state_weights(self, weights, set_epoch=True):
        super().set_full_state_weights(weights, set_epoch=set_epoch)
        cv = self.central_value_net
        if 'assymetric_vf_nets' in weights:
            cv.load_state_dict(weights['assymetric_vf_nets'])
        osd = weights.get('assymetric_vf_optimizer')
        if osd:
            lr, step = cv.load_optimizer_state_dict(osd)
            cv.lr = float(lr)
            cv.opt_state.copy_(adam_opt_state(cv.lr, step))
