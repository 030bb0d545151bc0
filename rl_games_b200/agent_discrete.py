"""Discrete-action PPO agent on the fp32 CUDA kernels -- SURVEY.md 8a row a15 (reference: algos_torch/a2c_discrete.py
DiscreteA2CAgent + common/a2c_common.py:1205-1359 DiscreteA2CBase, models.py:62-125 ModelA2C, network_builder.py A2CBuilder with a
``discrete`` space, optionally ``separate: True`` actor/critic trunks, optional action masks).

STATUS: parity-green on a B200 (round 2, ``tests/test_discrete_gpu.py``) against a CPU oracle that is pinned to the reference
(oracle/ppo_discrete_oracle.py, tests/golden/agent_discrete*.pt).  Everything except the two categorical kernels
(csrc/discrete.cu) reuses the kernels of the continuous path: linear_fwd / linear_bwd_* / reduce_splits (mlp_simt.cu), gae_fused, prepare_batch, moments_update,
mask_inv_counts (stats.cu, gae.cu), post_step (rollout.cu), adam_step (adam.cu).  The parameter arena is ``model.FlatArena`` and the
fp32 trunks are ``model.mlp_forward`` / ``mlp_backward``, shared with the central-value critic; config parsing, the outer train() loop,
summary scalars, the pooled normaliser sync and checkpoints are ``agent_base.A2CBase``, shared with the continuous agent.

Scope of this first edition: one GPU, eager launches (no CUDA graph), flat Box observations, ``Discrete(K)`` or multi-discrete
``Tuple(Discrete(K_j))`` action spaces (K_j <= 64, <= 8 heads), no RNN, no central value.  The scheduler steps once per MINI-EPOCH on the mean KL like the reference
(a2c_common.py:1265-1272), which costs one host sync per mini-epoch.
"""
import time

import numpy as np
import torch
import torch.distributed as dist

from . import ops
from .agent_base import A2CBase
from .model import FlatArena, _RunningStats, _model_call, adam_opt_state, check_network_params, mlp_backward, mlp_forward


class DiscreteModel(FlatArena):
    """Flat fp32 parameter arena of A2CBuilder.Network for a discrete space.  Arena order: actor trunk, [critic trunk], fused head
    W_head [1 + K, Hl] (row 0 = value, rows 1.. = logits) and b_head [1 + K]; ``_param_views`` lists the tensors in the reference's
    ``model.parameters()`` order (actor_mlp.*, critic_mlp.*, value.*, logits.*) for state dicts and the index-keyed Adam state."""

    __call__ = _model_call

    def __init__(self, network_params, obs_dim, n_actions, device, normalize_input, normalize_value, head_sizes=None):
        self.head_sizes = list(head_sizes) if head_sizes else None          # multi-discrete: one logits head per Tuple component
        check_network_params(network_params)
        mlp = network_params['mlp']
        self.units = list(mlp['units'])
        if not self.units:
            raise NotImplementedError('empty MLP')
        self.activation = mlp.get('activation', 'relu')
        if self.activation not in ops.ACT:
            raise NotImplementedError(f'activation {self.activation}')
        self.act_id = ops.ACT[self.activation]
        if mlp.get('initializer', {'name': 'default'}).get('name', 'default') != 'default':
            raise NotImplementedError("only the 'default' mlp initializer is mirrored for discrete models")
        for k in ('cnn', 'rnn'):
            if k in network_params:
                raise NotImplementedError(f"'{k}' networks are not supported by the discrete B200 agent yet")
        self.separate = bool(network_params.get('separate', False))
        self.D, self.K = int(obs_dim), int(n_actions)
        self.device = torch.device(device)
        self.normalize_input, self.normalize_value = bool(normalize_input), bool(normalize_value)
        sizes, ins = [], self.D
        for i, u in enumerate(self.units):
            sizes += [(f'Wa{i}', (u, ins)), (f'ba{i}', (u,))]
            ins = u
        if self.separate:
            ins = self.D
            for i, u in enumerate(self.units):
                sizes += [(f'Wc{i}', (u, ins)), (f'bc{i}', (u,))]
                ins = u
        self.Hl = ins
        sizes += [('W_head', (1 + self.K, ins)), ('b_head', (1 + self.K,))]
        self._build_arena(sizes, self.device)
        self._default_init()
        self.running_mean_std = _RunningStats(self.D, self.device) if self.normalize_input else None
        self.value_mean_std = _RunningStats(1, self.device) if self.normalize_value else None

    def trunk(self, which):
        return self.layers('a' if which == 'actor' or not self.separate else 'c', len(self.units))

    def _param_views(self, arena=None):
        out = []
        for p in (['a', 'c'] if self.separate else ['a']):
            for i in range(len(self.units)):
                out += [self.view(f'W{p}{i}', arena), self.view(f'b{p}{i}', arena)]
        wh, bh = self.view('W_head', arena), self.view('b_head', arena)
        out += [wh[:1], bh[:1]]
        if self.head_sizes is None:
            return out + [wh[1:], bh[1:]]
        off = 1
        for k in self.head_sizes:          # ModuleList of heads: logits.{j}.weight / bias (network_builder.py:304-305)
            out += [wh[off:off + k], bh[off:off + k]]
            off += k
        return out

    def param_names(self):
        names = []
        for pre in (['actor_mlp', 'critic_mlp'] if self.separate else ['actor_mlp']):
            for i in range(len(self.units)):
                names += [f'a2c_network.{pre}.{2 * i}.weight', f'a2c_network.{pre}.{2 * i}.bias']
        names += ['a2c_network.value.weight', 'a2c_network.value.bias']
        if self.head_sizes is None:
            return names + ['a2c_network.logits.weight', 'a2c_network.logits.bias']
        for j in range(len(self.head_sizes)):
            names += [f'a2c_network.logits.{j}.weight', f'a2c_network.logits.{j}.bias']
        return names

class DiscreteA2CAgent(A2CBase):
    def __init__(self, base_name, params):
        config = params['config']
        # options of the reference agent that change what a run does and are not built for the discrete path: refuse, never ignore
        for key, bad in (('normalize_rms_advantage', bool(config.get('normalize_rms_advantage', False))),
                         ('epochs_between_resets', config.get('epochs_between_resets', 0) > 0),
                         ('self_play', config.get('self_play_config') is not None or bool(config.get('self_play', False)))):
            if bad:
                raise NotImplementedError(f'{key} is not built for the discrete B200 agent')
        if config.get('multi_gpu_sync_stats_mode', 'pooled') != 'pooled':
            raise NotImplementedError("multi_gpu_sync_stats_mode: only 'pooled' for the discrete agent")
        if config.get('central_value_config') is not None:
            raise NotImplementedError('central_value_config')
        # multi-GPU: the per-minibatch gradient exchange is an NCCL all-reduce of the flat gradient in front of the Adam kernel (which
        # applies 1/world), the scheduler sees the rank-mean KL
        super().__init__(base_name, params)
        if self.value_size != 1:
            raise NotImplementedError('value_size > 1')
        action_space = self.env_info['action_space']
        kind = type(action_space).__name__          # a2c_common.py:1211-1224
        if kind == 'Discrete':
            self.head_sizes, self.actions_num, self.is_multi_discrete = None, int(action_space.n), False
        elif kind == 'Tuple':
            self.head_sizes = [int(a.n) for a in action_space]
            self.actions_num, self.is_multi_discrete = sum(self.head_sizes), True      # width of the concatenated logits
            if len(self.head_sizes) > 8:
                raise NotImplementedError('more than 8 heads in a multi-discrete space')
        else:
            raise ValueError(f'Unsupported action space type for DiscreteA2CBase: {type(action_space)}')
        self.is_discrete = True
        if max(self.head_sizes or [self.actions_num]) > 64:
            raise NotImplementedError('more than 64 actions in one discrete head')
        self.use_action_masks = bool(config.get('use_action_masks', False))
        self.model = DiscreteModel(self.network_params, self.obs_shape[0], self.actions_num, self.device_t, self.normalize_input,
                                   self.normalize_value, head_sizes=self.head_sizes)
        self.value_mean_std = self.model.value_mean_std
        self.rng_seed = int(config.get('b200_rng_seed', params.get('seed', 0) or 0))
        self.is_tensor_obses = True
        self.algo_observer.after_init(self)

    # =============================================================================== allocation
    def init_tensors(self):
        if self._tensors_ready:
            return
        H, N, D, K, m, mb = self.horizon_length, self.num_actors, self.obs_shape[0], self.actions_num, self.model, self.minibatch_size
        dev = self.device_t
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)   # noqa: E731
        self.obses = f(H, N, D)
        self.actions = (torch.zeros(H, N, len(self.head_sizes), dtype=torch.int64, device=dev) if self.head_sizes
                        else torch.zeros(H, N, dtype=torch.int64, device=dev))
        self.neglogpacs, self.values, self.rewards = f(H, N), f(H, N), f(H, N)
        self.dones_buf = torch.zeros(H, N, dtype=torch.uint8, device=dev)
        self.action_masks = torch.ones(H, N, K, dtype=torch.uint8, device=dev) if self.use_action_masks else None
        self.valid = torch.ones(H, N, dtype=torch.float32, device=dev) if self.mask_autoreset_rows else None
        self.advs, self.returns = f(H, N), f(H, N)
        self.old_values_n, self.returns_n, self.advs_n = f(H, N), f(H, N), f(H, N)
        self.last_values = f(N)
        self.ep_state = f(3, N)
        self.dones = torch.ones(N, dtype=torch.uint8, device=dev)
        self.prev_dones = f(N) if self.mask_autoreset_rows else None
        self.meter = torch.zeros(8, dtype=torch.float64, device=dev)
        self.rng_epoch = torch.zeros(1, dtype=torch.int64, device=dev)
        L = len(m.units)
        # rollout / training activations of the actor trunk (and the critic trunk when separate), head buffers
        self.r_a = [f(N, u) for u in m.units]
        self.r_c = [f(N, u) for u in m.units] if m.separate else self.r_a
        self.t_a = [f(mb, u) for u in m.units]
        self.t_c = [f(mb, u) for u in m.units] if m.separate else self.t_a
        self.d_a = [f(mb, u) for u in m.units]
        self.d_c = [f(mb, u) for u in m.units] if m.separate else self.d_a
        self.r_head, self.t_head, self.d_head = f(N, 1 + K), f(mb, 1 + K), f(mb, 1 + K)
        self.n_splits = max(1, min(64, mb // 256))
        self.part = f(self.n_splits, m.num_params)
        self.grad = f(m.num_params)
        self.loss_partials = torch.zeros((mb + 255) // 256, 8, dtype=torch.float64, device=dev)
        self.gae_partials = torch.zeros(max(64, (N + 63) // 64), 8, dtype=torch.float64, device=dev)
        self.inv_counts = f(self.num_minibatches) if self.mask_autoreset_rows else None
        self.mom_scratch = torch.zeros(148 * 4 * 2 * D, dtype=torch.float64, device=dev)
        self.post_scratch = torch.zeros(((N + 255) // 256) * 4, dtype=torch.float64, device=dev)
        self.counters = torch.zeros(4, dtype=torch.int32, device=dev)
        self.opt_state = adam_opt_state(self.last_lr, 0).to(dev)
        self.adam_stats = f(16)
        self.opt_cfg = ops.OptCfg(0.9, 0.999, 1e-8, float(self.weight_decay), float(self.grad_norm), 0.0, 1e-6, 1e-2, 1.5,
                                  1.0 / self.world_size, int(bool(self.truncate_grads)), 0)
        rs = self.rewards_shaper
        self.shaper_cfg = ops.ShaperCfg(float(rs.scale_value), float(rs.shift_value), float(rs.min_val), float(rs.max_val),
                                        float(self.gamma), int(bool(rs.log_val)), int(bool(self.value_bootstrap)))
        self._tensors_ready = True
        assert L >= 1

    # =============================================================================== env plumbing (tensor envs on the device)
    def _to_dev(self, x, dtype=None):
        t = x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x))
        t = t.to(self.device_t)
        return t if dtype is None or t.dtype == dtype else t.to(dtype)

    def env_reset(self):
        o = self.vec_env.reset()
        o = o['obs'] if isinstance(o, dict) else o
        return self._to_dev(o, torch.float32).contiguous()

    def env_step(self, actions):
        o, rewards, dones, infos = self.vec_env.step(actions)
        o = o['obs'] if isinstance(o, dict) else o
        return self._to_dev(o, torch.float32).contiguous(), self._to_dev(rewards, torch.float32), self._to_dev(dones), infos

    # =============================================================================== forward pieces
    def _norm(self):
        r = self.model.running_mean_std
        return (r.mean_f32, r.std_f32) if self.normalize_input else (None, None)

    def _forward(self, x, a_acts, c_acts, head, M, rows_per_chunk=None, chunk_stride=0):
        """actor trunk, [critic trunk], heads over M rows of x; returns _head_views(head, M)"""
        m = self.model
        for which, acts in (('actor', a_acts), ('critic', c_acts))[:1 + m.separate]:
            mlp_forward(m.trunk(which), x, acts, m.act_id, M, m.D, self._norm(), rows_per_chunk, chunk_stride)
        self._heads(a_acts[-1], c_acts[-1], head, M)
        return self._head_views(head, M)

    def _heads(self, a_last, c_last, head, M):
        """head[:, 0] = value, head[:, 1:] = logits (one GEMM when the trunk is shared)"""
        m = self.model
        wh, bh = m.view('W_head'), m.view('b_head')
        if not m.separate:
            ops.linear_fwd(a_last, wh, bh, head, 0, M=M)
            return
        # separate trunks: two skinny GEMMs into strided halves of the same head buffer is not expressible with linear_fwd's dense
        # output, so the value and the logits go to their own dense buffers
        ops.linear_fwd(c_last, wh[:1], bh[:1], self._val_buf(M), 0, M=M)
        ops.linear_fwd(a_last, wh[1:], bh[1:], self._logit_buf(M), 0, M=M)

    def _val_buf(self, M):
        if not hasattr(self, '_vb'):
            self._vb = {}
        return self._vb.setdefault(M, torch.zeros(M, 1, dtype=torch.float32, device=self.device_t))

    def _logit_buf(self, M):
        if not hasattr(self, '_lb'):
            self._lb = {}
        return self._lb.setdefault(M, torch.zeros(M, self.actions_num, dtype=torch.float32, device=self.device_t))

    def _head_views(self, head, M):
        """(logits, ld, value, value_ld) of the forward buffers for M rows"""
        K = self.actions_num
        if self.model.separate:
            return self._logit_buf(M), K, self._val_buf(M), 1
        return head[:, 1:], K + 1, head, K + 1

    # =============================================================================== rollout
    def play_steps(self, u=None):
        """a2c_common.py:985-1069 for a discrete space; u: optional [H + 1, N] uniform tape (tests) -- else Philox."""
        self.init_tensors()
        H, N, K, m = self.horizon_length, self.num_actors, self.actions_num, self.model
        vm = m.value_mean_std
        step_time = 0.0
        for t in range(H):
            obs = self.obs
            self.obses[t].copy_(obs)
            masks = None
            if self.use_action_masks:          # a2c_common.py:995-997
                masks = self._to_dev(self.vec_env.get_action_masks()).to(torch.uint8).contiguous()
                self.action_masks[t].copy_(masks)
            lg, ld, vl, vld = self._forward(obs, self.r_a, self.r_c, self.r_head, N)
            ops.categorical_sample(lg, ld, K, vl, vld, masks, None if u is None else u[t].contiguous(), self.rng_seed, self.rng_epoch, t,
                                   None if vm is None else vm.running_mean, None if vm is None else vm.running_var, self.normalize_value,
                                   self.actions[t], self.neglogpacs[t], self.values[t], self.dones, self.dones_buf[t], self.prev_dones,
                                   None if self.valid is None else self.valid[t], N, head_sizes=self.head_sizes)
            t0 = time.perf_counter()
            self.obs, rewards, dones, infos = self.env_step(self.actions[t])
            step_time += time.perf_counter() - t0
            tout = infos.get('time_outs') if (self.value_bootstrap and isinstance(infos, dict)) else None
            if tout is not None:
                tout = self._to_dev(tout)
            ops.post_step(rewards, dones, tout, self.values[t], None if self.valid is None else self.valid[t], self.rewards[t],
                          self.dones, self.prev_dones, self.ep_state, self.meter, self.games_to_track, self.post_scratch,
                          self.counters[0:1], N, self.shaper_cfg)
            if getattr(self.algo_observer, 'wants_done_indices', True):
                self.algo_observer.process_infos(infos, self.dones.nonzero(as_tuple=False))
            elif getattr(self.algo_observer, 'wants_infos', False):
                self.algo_observer.process_infos(infos, None)
        # get_values (a2c_common.py:603-626): the reference's forward samples here too; only the value is used
        lg, ld, vl, vld = self._forward(self.obs, self.r_a, self.r_c, self.r_head, N)
        ops.categorical_sample(None, ld, K, vl, vld, None, None, 0, None, 0, None if vm is None else vm.running_mean,
                               None if vm is None else vm.running_var, self.normalize_value, None, None, self.last_values, None, None,
                               None, None, N, values_only=True)
        ops.bump_u64(self.rng_epoch)
        self._meter_cache = None
        return step_time

    def _gae_and_prepare(self):
        m = self.model
        nb = ops.gae_fused(self.rewards, self.values, self.dones_buf, self.last_values, self.dones, self.valid, self.advs, self.returns,
                           self.gae_partials, self.gamma, self.tau)
        vm = m.value_mean_std
        dummy = getattr(self, '_dummy_vms', None)
        if vm is None and dummy is None:
            dummy = self._dummy_vms = _RunningStats(1, self.device_t)
        s = vm if vm is not None else dummy
        ops.prepare_batch(self.values, self.returns, self.valid, self.gae_partials, nb, s.running_mean, s.running_var, s.count,
                          self.old_values_n, self.returns_n, self.advs_n, self.normalize_value, self.normalize_advantage)
        if self.mask_autoreset_rows:
            ops.mask_inv_counts(self.valid, self.horizon_length, self.num_actors, self.envs_per_mb, self.inv_counts)

    # =============================================================================== update
    def _minibatch_update(self, i):
        """calc_gradients (a2c_discrete.py:121-209) + trancate_gradients_and_step for minibatch i; returns a device row
        [a_loss, c_loss, entropy, kl] (masked means)."""
        m, H, N, K = self.model, self.horizon_length, self.num_actors, self.actions_num
        epm, mb, P, S = self.envs_per_mb, self.minibatch_size, self.model.num_params, self.n_splits
        e0 = i * epm
        x = self.obses[0, e0:]
        if self.normalize_input:      # set_train() re-arms the obs normaliser before every minibatch (see oracle/ppo_oracle.py)
            r = m.running_mean_std
            ops.moments_update(x, m.D, epm, H, N, r.running_mean, r.running_var, r.count, r.mean_f32, r.std_f32, self.mom_scratch,
                               self.counters[1:2])
        lg, ld, vl, vld = self._forward(x, self.t_a, self.t_c, self.t_head, mb, rows_per_chunk=epm, chunk_stride=N)
        if m.separate:
            d_lg, d_ld, d_vl, d_vld = self._dl_buf(), K, self._dv_buf(), 1
        else:
            d_lg, d_ld, d_vl, d_vld = self.d_head[:, 1:], K + 1, self.d_head, K + 1
        cfg = ops.CatLossCfg(float(self.e_clip), float(self.critic_coef), float(self.entropy_coef), int(bool(self.clip_value)),
                             int(bool(self.use_smooth_clamp)), int(bool(self.ppo)))
        nb = ops.categorical_loss(lg, ld, K, vl, vld, self.actions[0, e0:], None if self.action_masks is None else self.action_masks[0, e0:],
                                  self.old_values_n[0, e0:], self.returns_n[0, e0:], self.neglogpacs[0, e0:], self.advs_n[0, e0:],
                                  None if self.valid is None else self.valid[0, e0:], epm, N, mb, cfg,
                                  None if self.inv_counts is None else self.inv_counts[i:i + 1], d_lg, d_ld, d_vl, d_vld,
                                  self.loss_partials, head_sizes=self.head_sizes)
        stats = self.loss_partials[:nb, :4].sum(dim=0).float()
        # ---- backward through the heads and the trunk(s): split partial gradients, then one reduction ----
        off_wh, _ = m.layout['W_head']
        off_bh, _ = m.layout['b_head']
        if m.separate:
            Hl = m.Hl
            ops.linear_bwd_weight(d_vl, self.t_c[-1], self.part[0, off_wh:], self.part[0, off_bh:], Hl, 1, S, M=mb, split_stride=P)
            ops.linear_bwd_weight(d_lg, self.t_a[-1], self.part[0, off_wh + Hl:], self.part[0, off_bh + 1:], Hl, K, S, M=mb, split_stride=P)
            wh = m.view('W_head')
            ops.linear_bwd_data(d_vl, wh[:1], self.t_c[-1], self.d_c[-1], m.act_id, M=mb)
            ops.linear_bwd_data(d_lg, wh[1:], self.t_a[-1], self.d_a[-1], m.act_id, M=mb)
        else:
            ops.linear_bwd_weight(self.d_head, self.t_a[-1], self.part[0, off_wh:], self.part[0, off_bh:], m.Hl, 1 + K, S, M=mb,
                                  split_stride=P)
            ops.linear_bwd_data(self.d_head, m.view('W_head'), self.t_a[-1], self.d_a[-1], m.act_id, M=mb)
        for which, acts, dacts in (('actor', self.t_a, self.d_a), ('critic', self.t_c, self.d_c))[:1 + m.separate]:
            mlp_backward(m.trunk(which), self.part, x, acts, dacts, m.act_id, mb, m.D, self._norm(), epm, N)
        ops.reduce_splits(self.part, self.grad, P, S, split_stride=P)
        if self.multi_gpu:          # a2c_common.py:493-509 (the Adam kernel applies the 1/world scale)
            dist.all_reduce(self.grad, op=dist.ReduceOp.SUM)
        ops.adam_step(m.flat, self.grad, m.exp_avg, m.exp_avg_sq, self.opt_state, None, self.opt_cfg, self.adam_stats, self.counters[2:3],
                      n=P)
        return stats

    def _dl_buf(self):
        if not hasattr(self, '_dlb'):
            self._dlb = torch.zeros(self.minibatch_size, self.actions_num, dtype=torch.float32, device=self.device_t)
        return self._dlb

    def _dv_buf(self):
        if not hasattr(self, '_dvb'):
            self._dvb = torch.zeros(self.minibatch_size, 1, dtype=torch.float32, device=self.device_t)
        return self._dvb

    def train_epoch(self, u=None):
        """DiscreteA2CBase.train_epoch (a2c_common.py:1233-1289): returns the reference's tuple."""
        self.init_tensors()
        if self.obs is None:
            self.obs = self.env_reset()
        t0 = time.perf_counter()
        step_time = self.play_steps(u)
        self._gae_and_prepare()
        self._sync()
        t1 = time.perf_counter()
        self.curr_frames = self.batch_size
        self.algo_observer.after_steps()
        rows, kls = [], []
        for _ in range(self.mini_epochs_num):
            lr_used = self.last_lr          # what train_actor_critic returns for the minibatches of this mini-epoch (:1265, :1289)
            ep = [self._minibatch_update(i) for i in range(self.num_minibatches)]
            rows += ep
            av_kl = torch.stack([r[3] for r in ep]).mean()          # torch_ext.mean_list
            if self.multi_gpu:                                      # a2c_common.py:1272-1274
                dist.all_reduce(av_kl, op=dist.ReduceOp.SUM)
                av_kl = av_kl / self.world_size
            self.last_lr, self.entropy_coef = self.scheduler.update(self.last_lr, self.entropy_coef, self.epoch_num, self.frame,
                                                                    av_kl.item())                  # one host sync per mini-epoch (:1271)
            self.opt_state[0] = self.last_lr                        # update_lr
            kls.append(av_kl)
        self.sync_running_stats()
        self._sync()
        t2 = time.perf_counter()
        st = torch.stack(rows)
        self.last_stats = st
        a_losses, c_losses, entropies = list(st[:, 0]), list(st[:, 1]), list(st[:, 2])
        return step_time, t1 - t0, t2 - t1, t2 - t0, a_losses, c_losses, entropies, kls, lr_used, 1.0

    # =============================================================================== train loop / checkpoints (agent_base.A2CBase)
    def _on_train_start(self):
        self.mean_rewards = -float('inf')      # last_mean_rewards (best-ever watermark) is deliberately NOT reset here

    def _optimizer_lr(self):
        return float(self.opt_state.cpu()[0])

    def _restore_optimizer(self, lr, step):
        # the restored lr drives the optimiser until the next scheduler step (end of the first mini-epoch), which continues from this
        # agent's own last_lr
        self.opt_state.copy_(adam_opt_state(float(lr) if lr is not None else self.last_lr, step))
