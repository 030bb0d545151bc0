"""B200-native continuous PPO agent behind the reference's plugin surface.

Same constructor (``A2CAgent(base_name, params)``), config keys / defaults and public methods as
``rl_games.algos_torch.a2c_continuous.A2CAgent`` + ``rl_games.common.a2c_common.ContinuousA2CBase``
(a2c_common.py:170-491 config parsing, :985-1069 play_steps, :1517-1584 train_epoch, :1586-1660
prepare_dataset, :1662-1782 train; a2c_continuous.py:136-234 calc_gradients), but the hot loop is a
sequence of hand-written sm_100a kernels over one time-major experience arena:

    rollout step t:   [obs copy] -> MLP fwd (norm fused) -> policy_head_sample -> env.step -> post_step
    epoch end:        values_only fwd -> gae_fused (+returns +moment partials) -> prepare_batch
    minibatch i:      obs moments+merge -> MLP fwd -> ppo_head_loss -> finalize -> wgrad/dgrad chain ->
                      split reduce -> [NCCL all-reduce of the flat grad (+KL slot)] -> adam_step (+ on-device
                      adaptive-KL LR schedule)

No tensor is ever transposed/flattened: the reference's flat sample index env*H+t (swap_and_flatten01,
a2c_common.py:33-40) and minibatch slices (datasets.py:75-82) are honoured as an index mapping --
minibatch i = envs [i*mb/H, (i+1)*mb/H) x all t.  The whole update phase (mini_epochs x num_minibatches)
is captured in one CUDA graph; no .item()/nonzero() host syncs remain inside an epoch.

Config parsing, device / multi-GPU / env setup, the outer train() loop, summary scalars, the cross-rank normaliser sync and the
checkpoint dict are ``agent_base.A2CBase``, shared with the discrete agent; this module adds the continuous keys, the kernels' arenas and
schedules, the bounds-loss scalar and the checkpoint extras (advantage EMA state, the one-step hold of a restored optimizer lr).
"""
import time

import numpy as np
import torch
import torch.distributed as dist

from . import ops
from .agent_base import A2CBase
from .common import IdentityScheduler
from .model import B200Model, adam_opt_state


def swap_and_flatten01(arr):
    """a2c_common.py:33-40 -- only used to hand reference-layout views to callers (tests, observers)."""
    if arr is None:
        return arr
    s = arr.size()
    return arr.transpose(0, 1).reshape(s[0] * s[1], *s[2:])


def rescale_actions(low, high, action):
    """a2c_common.py:144-148"""
    d = (high - low) / 2.0
    m = (high + low) / 2.0
    return action * d + m


class _Dataset:
    """datasets.PPODataset look-alike (datasets.py:7-95): len() minibatches, [i] -> dict of reference-layout
    COPIES of minibatch i (flat order env*H+t) tagged with its index so train_actor_critic() can run the
    fused kernels on the arena rows the slice denotes."""

    def __init__(self, agent):
        self.a = agent
        self.values_dict = None

    def __len__(self):
        return self.a.num_minibatches

    def update_values_dict(self, d):
        self.values_dict = d

    def __getitem__(self, i):
        a = self.a
        e0, e1 = i * a.envs_per_mb, (i + 1) * a.envs_per_mb
        fl = lambda t: swap_and_flatten01(t[:, e0:e1])   # noqa: E731
        d = {'old_values': fl(a.old_values_n).unsqueeze(1), 'old_logp_actions': fl(a.neglogpacs),
             'advantages': fl(a.advs_n), 'returns': fl(a.returns_n).unsqueeze(1), 'actions': fl(a.actions),
             'obs': fl(a.obses), 'dones': fl(a.dones_buf), 'mu': fl(a.mus), 'sigma': fl(a.sigmas), '_mb_index': i}
        if a.mask_autoreset_rows:
            d['rnn_masks'] = fl(a.valid)
        return d


class A2CAgent(A2CBase):
    def __init__(self, base_name, params):
        config = params['config']
        # options of A2CBase that change what a run does and are not built here: refuse, never ignore
        if config.get('epochs_between_resets', 0) > 0:
            raise NotImplementedError('epochs_between_resets (forced env resets, a2c_common.py:553-556)')
        if config.get('self_play_config') is not None or config.get('self_play', False):
            raise NotImplementedError('self-play (SelfPlayManager) is outside the B200 hot path')
        model_name = params.get('model', {}).get('name', 'continuous_a2c_logstd')
        if model_name != 'continuous_a2c_logstd':
            raise NotImplementedError(f"model '{model_name}': only continuous_a2c_logstd is on the B200 hot path")
        if config.get('use_action_masks', False):
            raise NotImplementedError('action masks are a discrete-PPO feature')
        if config.get('central_value_config') is not None:
            raise NotImplementedError('central_value_config is served by rl_games_b200.agent_cv.A2CAgentCV: build the agent through '
                                      'rl_games_b200.register(runner) / rl_games_b200.runner.continuous_agent, which pick it')
        super().__init__(base_name, params)
        self.schedule_type = config.get('schedule_type', 'per_minibatch')
        if self.schedule_type == 'legacy':
            self.schedule_type = 'per_minibatch'
        if self.is_adaptive_lr and self.schedule_type not in ('per_minibatch', 'standard'):
            raise NotImplementedError("adaptive lr_schedule with schedule_type=%r: 'per_minibatch' (the default) and 'standard' "
                                      "(one step per mini-epoch) run on the device scheduler" % self.schedule_type)
        # EMA advantage normaliser (a2c_common.py:369, :473-475): GeneralizedMovingStats((1,), decay=adv_rms_momentum), 'mean_std'
        self.normalize_rms_advantage = bool(config.get('normalize_rms_advantage', False)) and self.normalize_advantage
        self.adv_rms_momentum = float(config.get('adv_rms_momentum', 0.5))
        # None (key absent) = the reference's 'auto' (a2c_common.py:427-429): resolved once the model geometry is known
        self.mixed_precision = config.get('mixed_precision', None)
        self.is_tensor_obses = False
        self.zero_rnn_on_done = config.get('zero_rnn_on_done', True)

        # ---- ContinuousA2CBase (a2c_common.py:1484-1497) ----
        self.is_discrete = False
        action_space = self.env_info['action_space']
        self.actions_num = action_space.shape[0]
        self.bounds_loss_coef = config.get('bounds_loss_coef', None)
        self.bound_loss_type = config.get('bound_loss_type', 'bound')
        self.clip_actions = config.get('clip_actions', True)
        self.actions_low = torch.from_numpy(np.asarray(action_space.low).copy()).float().to(self.device_t)
        self.actions_high = torch.from_numpy(np.asarray(action_space.high).copy()).float().to(self.device_t)

        # ---- A2CAgent (a2c_continuous.py:27-76) ----
        self.model = B200Model(self.network_params, self.obs_shape[0], self.actions_num, self.device_t,
                               self.normalize_input, self.normalize_value, self.value_size)
        self.value_mean_std = self.model.value_mean_std if self.normalize_value else None
        # precision mode: mixed_precision True -> bf16 tcgen05 kernels (mlp_tc.cu); False -> fp32 CUDA-core kernels (mlp_simt.cu).
        # An explicit True is never downgraded (unsupported geometry raises); an ABSENT key is the reference's 'auto' (bf16 where the
        # hardware supports it, a2c_common.py:427-429) and resolves to the tcgen05 path where this build has kernels for the
        # geometry, else to fp32 (a HIGHER precision than the reference's default), saying so once.
        self.is_rnn = self.model.is_rnn()
        # wide observations (64 < obs <= 256): layer 1 runs in kernels of its own (l1_fwd_tc / l1_wgrad_tc)
        allow_wide = True
        # tcgen05 kernels: three hidden layers that fit the compiled tile widths (u1 <= 256, u2 <= 128, u3 <= 64; narrower layers are
        # zero-padded), elu / relu / tanh, obs <= 256, <= 15 actions; anything else runs on the fp32 kernels
        tc_ok = self.model.activation in ('elu', 'relu', 'tanh') and \
            ops.tc_supported(self.model.D, self.model.units, self.actions_num, allow_wide)
        # (a sigma floor -- min_sigma > 0 -- is applied outside the kernels on the log-std vector they read; the fused kernels take the raw
        #  parameter from the packed arena, so such policies run layer by layer.  Separate actor / critic trunks need their gradient mask
        #  applied between the split reduction and the optimiser, which the fused tail does in one launch: layer by layer as well)
        fused_ok = tc_ok and not self.is_rnn and getattr(self.model, 'min_sigma', 0.0) == 0 and not getattr(self.model, 'separate', False)
        if self.mixed_precision is None:
            self.mixed_precision = fused_ok
            if not self.mixed_precision and self.global_rank == 0:
                print(f'b200: mixed_precision not set -> fp32 kernels for this geometry (obs={self.model.D}, units={self.model.units}, '
                      f'actions={self.actions_num}, activation={self.model.activation}{", rnn" if self.is_rnn else ""}); mixed_precision: True runs it '
                      f'on the tensor cores layer by layer; the FUSED bf16 tcgen05 kernels cover obs<=256, three-layer MLPs up to [256,128,64] '
                      f'with elu / relu / tanh, actions<=15')
        if self.is_rnn:
            if self.horizon_length % self.seq_length != 0:
                raise ValueError(f"Horizon length ({self.horizon_length}) must be divisible by sequence length ({self.seq_length})")
            if not self.zero_rnn_on_done:
                raise NotImplementedError('zero_rnn_on_done: False is not on the B200 hot path')
        # mixed_precision: True -> the fused tcgen05 MLP kernels where they have the geometry (use_tc), else the SAME host composition as the
        # fp32 path with every GEMM on the tensor cores (gemm_tc: bf16 operands, fp32 accumulate -- gemm_tc.cu): LSTM policies (gate GEMMs,
        # BPTT), MLPs wider / deeper than the fused tiles.  The reference's autocast covers nn.LSTM and nn.Linear alike (a2c_continuous.py:173).
        self.use_tc = bool(self.mixed_precision) and fused_ok
        self.gemm_tc = bool(self.mixed_precision) and not fused_ok
        self._lin_fwd = ops.linear_fwd_tc if self.gemm_tc else ops.linear_fwd
        self._lin_bwd = ops.linear_bwd_data_tc if self.gemm_tc else ops.linear_bwd_data
        self._lin_bww = ops.linear_bwd_weight_tc if self.gemm_tc else ops.linear_bwd_weight
        self.tc_wide = self.use_tc and ops.tc_kind(self.model.D, self.model.units, self.actions_num) == 2
        # Rollout precision.  The reference evaluates the policy during the rollout OUTSIDE autocast (a2c_common.py:581-600: fp32 / TF32)
        # and only calc_gradients under bf16 autocast (a2c_continuous.py:173).  Default here: the rollout uses the same bf16 tcgen05
        # kernels as the update, so old_neglogp / old mu come from the SAME arithmetic the first mini-epoch re-evaluates (ratio == 1 at
        # the first minibatch, which the reference's mix does not give).  b200_rollout_fp32: True restores the reference's split: fp32
        # CUDA-core kernels for get_action_values / get_values, bf16 tensor cores for the update.
        self.rollout_fp32 = self.use_tc and bool(config.get('b200_rollout_fp32', False))
        if self.use_tc and config.get('b200_pipelined_wgrad', False) and (self.tc_wide or list(self.model.units) != [256, 128, 64]):
            raise NotImplementedError('b200_pipelined_wgrad is an option of the native resident-weights geometry (obs <= 64, MLP [256,128,64])')
        self.dataset = _Dataset(self)
        self.has_value_loss = True
        self.use_cuda_graph = bool(config.get('b200_cuda_graph', True))
        # NCCL all-reduces are stream-ordered and graph-capturable; opt-out knob for debugging
        self.graph_multi_gpu = bool(config.get('b200_cuda_graph_multi_gpu', True))
        self.rng_seed = int(config.get('b200_rng_seed', params.get('seed', 0) or 0)) + 7919 * self.global_rank
        self._graph_update = None
        self._graph_epoch = None
        self.train_result = None
        self.algo_observer.after_init(self)

    # =============================================================================== allocation
    def init_tensors(self):
        """a2c_common.py:634-660 + experience.py:330-398: one time-major arena, zero-initialised."""
        if self._tensors_ready:
            return
        H, N, D, A = self.horizon_length, self.num_actors, self.obs_shape[0], self.actions_num
        dev = self.device_t
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)   # noqa: E731
        self.obses = f(H, N, D)
        self.actions, self.mus, self.sigmas = f(H, N, A), f(H, N, A), f(H, N, A)
        self.neglogpacs, self.values, self.rewards = f(H, N), f(H, N), f(H, N)
        self.dones_buf = torch.zeros(H, N, dtype=torch.uint8, device=dev)
        self.valid = torch.ones(H, N, dtype=torch.float32, device=dev) if self.mask_autoreset_rows else None
        self.advs, self.returns = f(H, N), f(H, N)
        self.old_values_n, self.returns_n, self.advs_n = f(H, N), f(H, N), f(H, N)
        self.last_values = f(N)
        self.env_actions = f(N, A)
        # rl_games names (experience.py:372-398) -> arena views, for observers / tests
        self.tensor_dict = {'obses': self.obses, 'rewards': self.rewards.unsqueeze(2), 'values': self.values.unsqueeze(2),
                            'neglogpacs': self.neglogpacs, 'dones': self.dones_buf, 'actions': self.actions,
                            'mus': self.mus, 'sigmas': self.sigmas}
        # episode bookkeeping (a2c_common.py:662-666)
        self.ep_state = f(3, N)
        self.dones = torch.ones(N, dtype=torch.uint8, device=dev)
        self.prev_dones = f(N) if self.mask_autoreset_rows else None
        self.meter = torch.zeros(8, dtype=torch.float64, device=dev)
        self.rng_epoch = torch.zeros(1, dtype=torch.int64, device=dev)
        # workspaces
        m, mb = self.model, self.minibatch_size
        if self.rollout_fp32:
            self.ra = [f(N, u) for u in m.units]
        if not self.use_tc:
            self.ra = [f(N, u) for u in m.units]
            self.ta = [f(mb, u) for u in m.units]
            self.dA = [f(mb, u) for u in m.units]
            self.d_head = f(mb, A + 1)
        ops.set_pdl(self.config.get('b200_pdl', False))     # programmatic dependent launch: measured slower on c2 (profiles/r01_summary.md)
        if self.use_tc:
            self.n_splits = 148
            tb = ops.tc_tile_bytes(m.D, m.units, A)
            nt = (mb + 127) // 128
            u8 = lambda n: torch.zeros(n, dtype=torch.uint8, device=dev)   # noqa: E731
            self.wpack = u8(ops.tc_pack_bytes(m.D, m.units, A))
            # wide observations: the rollout's layer-1 kernel parks its a1 tiles (N rows) in the act1 buffer between the two launches
            nt1 = max(nt, (N + 127) // 128) if self.tc_wide else nt
            self.tc_act = [u8(nt1 * tb[0]), u8(nt * tb[1]), u8(nt * tb[2])]
            self.tc_l1_scratch = self.tc_act[0] if self.tc_wide else None
            self.tc_dhead, self.tc_delta2, self.tc_delta1 = u8(nt * tb[3]), u8(nt * tb[1]), u8(nt * tb[0])
            # normalised bf16 obs tiles: the training forward emits them, the backward's layer-1 weight-gradient MMAs TMA-load
            # them instead of re-reading and re-normalising the fp32 observations (b200_emit_xtile: False restores that); config
            # b200_pipelined_wgrad selects the two-stage-ring edition of the weight-gradient kernel (measured slower on c2)
            self.tc_pipelined_wgrad = bool(self.config.get('b200_pipelined_wgrad', False))
            want_xt = self.tc_pipelined_wgrad or bool(self.config.get('b200_emit_xtile', True))
            self.tc_xt = u8(nt * ops.tc_xtile_bytes(m.D, m.units, A)) if want_xt else None
            self.tc_offs = {k: m.layout[k][0] for k in ('W0', 'b0', 'W1', 'b1', 'W2', 'b2', 'W_head', 'b_head')}
            self.pack_table = ops.tc_pack_table(m.D, m.units, A, self.tc_offs)
            self.ta = self.dA = []
            if not self.rollout_fp32:
                self.ra = []
        elif self.gemm_tc:
            # layer-wise tensor-core GEMMs: a weight-gradient CTA owns a [128 x <=256] tile of dW and a row split; 16 splits keep the
            # c4 gate GEMM (16 tiles) at 256 CTAs while the split partials stay small (64 splits: 91 MB of partials per gate GEMM)
            self.n_splits = max(1, min(16, mb // 512))
            self.wbf = torch.empty(m.num_params, dtype=torch.bfloat16, device=dev)     # bf16 twin of the parameter arena (weight operands)
            import functools
            arena = (m.flat, self.wbf)
            self._lin_fwd = functools.partial(ops.linear_fwd_tc, bf16_arena=arena)
            self._lin_bwd = functools.partial(ops.linear_bwd_data_tc, bf16_arena=arena)
        else:
            self.n_splits = max(1, min(64, mb // 256))
        self.part_rows = self.n_splits * (self.seq_length if self.is_rnn else 1)
        # split-partial gradient rows; the tcgen05 path pads the row stride to 16 bytes so the reduction can use float4 loads
        self.part = f(self.part_rows, (m.num_params + 3) // 4 * 4 if self.use_tc else m.num_params)
        if self.is_rnn:
            Hd, T = m.rnn_units, self.seq_length
            S = mb // T
            self.rnn_h, self.rnn_c = f(N, Hd), f(N, Hd)                       # current states (a2c_common.py:652-655)
            # train-time reset flags: the buffer's dones, plus "entering the first real row after a filler reset row" on next_step envs
            self.rnn_dones_buf = torch.zeros(H, N, dtype=torch.uint8, device=dev) if self.mask_autoreset_rows else None
            self.rnn_h0, self.rnn_c0 = f(H // T, N, Hd), f(H // T, N, Hd)     # mb_rnn_states (:656-660), [num_seqs_per_env, N, hid]
            self.r_gates, self.r_tmp_h, self.r_tmp_c = f(N, 4 * Hd), f(N, Hd), f(N, Hd)
            self.t_gates, self.t_hin, self.t_cin, self.t_c = f(T, S, 4 * Hd), f(T, S, Hd), f(T, S, Hd), f(T, S, Hd)
            self.t_hdense, self.t_hmlp, self.t_dHmlp = f(S, Hd), f(mb, Hd), f(mb, Hd)
            self.t_dgates, self.t_dhin, self.t_dcin = f(S, 4 * Hd), f(S, Hd), f(2, S, Hd)
        self.gae_partials = torch.zeros((N + 63) // 64, 8, dtype=torch.float64, device=dev)
        self.loss_partials = torch.zeros(max((mb + 127) // 128, 148), ops.loss_partial_stride(), dtype=torch.float64, device=dev)
        self.n_updates = self.mini_epochs_num * self.num_minibatches
        self.stats = f(self.n_updates, 16)
        # comm buffer = flat gradient + 1 KL slot (one all-reduce per minibatch, a2c_common.py:493-509 + :1559-1561)
        self.comm = f(m.num_params + 1)
        m.grad = self.comm[:m.num_params]
        m.gW = [m.view(f'W{i}', m.grad) for i in range(len(m.units))]
        m.gb = [m.view(f'b{i}', m.grad) for i in range(len(m.units))]
        m.g_sigma = m.view('sigma', m.grad)
        m.gW_head, m.gb_head = m.view('W_head', m.grad), m.view('b_head', m.grad)
        self.kl_slot = self.comm[m.num_params:]
        self._gv = [dict(grad=m.grad, g_sigma=m.g_sigma, kl=self.kl_slot, comm=self.comm)] * 2
        self.fused_allreduce = False
        if self.multi_gpu and self.world_size > 1 and self.config.get('b200_fused_allreduce', True):
            self._setup_peer_comm()
        # lr, step, beta1^step, beta2^step, [KL sum, count of the running mini-epoch (schedule_type 'standard')], pad
        self.opt_state = adam_opt_state(self.last_lr, 0, slots=8).to(dev)
        self.entropy_coef_dev = torch.tensor([float(self.entropy_coef)], dtype=torch.float32, device=dev)
        # linear schedule (a2c_common.py:1557-1563): the reference steps the scheduler AFTER every minibatch with the current epoch
        # number, so the first minibatch of an epoch still runs on the previous epoch's (lr, entropy_coef) and the others on this
        # epoch's.  The host knows both before the epoch starts; the switch is two device-to-device copies after the first update.
        self._sched_switch = self.linear_lr and not isinstance(self.scheduler, IdentityScheduler)
        self.lr_next_dev = torch.tensor([self.last_lr], dtype=torch.float64, device=dev)
        self.ent_next_dev = torch.tensor([float(self.entropy_coef)], dtype=torch.float32, device=dev)
        self.inv_counts = f(self.num_minibatches) if self.mask_autoreset_rows else None
        self.mom_scratch = torch.zeros(1024 * 2 * D, dtype=torch.float64, device=dev)
        self.use_mb_moments = self.normalize_input and D % 4 == 0
        self.mbmom = torch.zeros(self.num_minibatches, 2 * D, dtype=torch.float64, device=dev)
        self.mb_shift = f(D)
        self.mb_counters = torch.zeros(self.num_minibatches, dtype=torch.int32, device=dev)
        if self.use_mb_moments:
            r = m.running_mean_std
            self._merge_structs = [ops.make_obs_merge(self.mbmom[i], self.mb_shift, D, mb, r.running_mean, r.running_var, r.count,
                                                      r.mean_f32, r.std_f32) for i in range(self.num_minibatches)]
        self.post_scratch = torch.zeros(((N + 255) // 256) * 4, dtype=torch.float64, device=dev)
        self.counters = torch.zeros(4, dtype=torch.int32, device=dev)
        if self.normalize_rms_advantage and not hasattr(self, 'adv_ema_state'):
            self.adv_ema_state = torch.zeros(2, dtype=torch.float32, device=dev)     # GeneralizedMovingStats: mean, mean of squares
            self.adv_ema_step = torch.ones(1, dtype=torch.int32, device=dev)
        self.ra_nrm = torch.zeros(148, dtype=torch.float64, device=dev)      # reduce_adam: per-CTA sum-of-squares partials
        self.ra_bar = torch.zeros(1, dtype=torch.int64, device=dev)          # reduce_adam: monotonic grid-barrier counter
        self.host_stats = torch.zeros(self.n_updates, 16, dtype=torch.float32).pin_memory()
        self.host_state = torch.zeros(10, dtype=torch.float64).pin_memory()
        self._events = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        self._build_cfg_structs()
        self.update_list = ['actions', 'neglogpacs', 'values', 'mus', 'sigmas']
        self.tensor_list = self.update_list + ['obses', 'states', 'dones']
        self._pinned = {}
        self._tensors_ready = True
        self._repack()

    def _setup_peer_comm(self):
        """CUDA-IPC mapped, parity-double-buffered gradient arenas + flag arrays for the fused all-reduce/Adam kernel."""
        if self.world_size > 8:
            return
        if self.n_updates % 2 != 0:
            return      # buffers alternate by update parity across epochs / graph replays: needs an even number of updates per epoch
        m, dev = self.model, self.device_t
        P = m.num_params
        S = ((P + 1 + 3) // 4) * 4
        # two exchange buffers (update parity), 8 per-rank flags (allreduce_adam), 8 x PEER_FLAG_STRIDE per-CTA flags (reduce_allreduce_adam)
        nbytes = 2 * S * 4 + 8 * 8 + 8 * ops.PEER_FLAG_STRIDE * 8
        base, handle = ops.ipc_alloc(nbytes)
        handles = [None] * self.world_size
        dist.all_gather_object(handles, handle)
        ptrs = [base if r == self.global_rank else ops.ipc_open(handles[r]) for r in range(self.world_size)]
        self._peer_keepalive = (base, ptrs)
        self.peer_table = ops.PeerTable([[p + par * S * 4 for p in ptrs] for par in (0, 1)], [p + 2 * S * 4 for p in ptrs],
                                        [p + 2 * S * 4 + 64 for p in ptrs])
        self.my_flags_ptr = base + 2 * S * 4
        self.my_cta_flags_ptr = base + 2 * S * 4 + 64
        # True = split reduction + all-reduce + Adam in ONE launch with per-CTA peer flags (reduce_allreduce_adam); default False =
        # reduce_finalize + allreduce_adam (two launches), measured faster at 2 GPUs: 3.71 vs 3.91 ms/epoch (profiles/r01_summary.md)
        self.fused_split_allreduce = bool(self.config.get('b200_fused_split_allreduce', False))
        self._gv = []
        for par in (0, 1):
            comm = ops.tensor_from_ptr(base + par * S * 4, P + 1, torch.float32, dev)
            grad = comm[:P]
            self._gv.append(dict(grad=grad, g_sigma=m.view('sigma', grad), kl=comm[P:], comm=comm))
        self.ar_seq = torch.zeros(1, dtype=torch.int64, device=dev)
        self.ar_red = torch.zeros(P + 1, dtype=torch.float32, device=dev)
        self.ar_nrm = torch.zeros(128, dtype=torch.float64, device=dev)
        self.ar_bar = torch.zeros(1, dtype=torch.int64, device=dev)
        self._ar_parity = 0
        self.fused_allreduce = True
        dist.barrier()

    def _merge_next(self, u):
        """obs-normaliser merge struct of update u+1's minibatch (performed by the optimiser kernel's last CTA), or None"""
        if self.use_mb_moments and u + 1 < self.n_updates and not getattr(self, '_compat_mode', False):
            return self._merge_structs[(u + 1) % self.num_minibatches]
        return None

    def _step_optimizer(self, u, gv, P, wpack=None, pack_table=None):
        """gradient exchange + clip + Adam (+ packed-weight refresh) for update u; the optimiser kernel's last CTA also performs the
        obs-normaliser update of the NEXT update's minibatch (the first one of an epoch is merged by _update_all)"""
        m = self.model
        mn = self._merge_next(u)
        self._set_sched_mode(u)
        if self.fused_allreduce:
            ops.allreduce_adam(self.peer_table, u & 1, self.global_rank, self.my_flags_ptr, self.ar_seq, self.ar_red, self.ar_nrm,
                               self.ar_bar, m.flat, m.exp_avg, m.exp_avg_sq, P, self.opt_state, self.opt_cfg, self.stats[u],
                               self.counters[2:3], wpack=wpack, pack_table=pack_table, merge_next=mn)
            if self.gemm_tc:
                ops.cast_bf16(m.flat, self.wbf)
            return
        if self.multi_gpu:
            dist.all_reduce(gv['comm'], op=dist.ReduceOp.SUM)
        ops.adam_step(m.flat, gv['grad'], m.exp_avg, m.exp_avg_sq, self.opt_state, gv['kl'], self.opt_cfg, self.stats[u],
                      self.counters[2:3], n=P, wpack=wpack, pack_table=pack_table, merge_next=mn)
        if self.gemm_tc:
            ops.cast_bf16(m.flat, self.wbf)

    def _set_sched_mode(self, u):
        """schedule_type 'standard' (a2c_common.py:1565-1571): the optimiser kernel of every minibatch adds its KL to the mini-epoch's
        running sum, the last one of the mini-epoch steps the scheduler on the mean.  The struct is read at launch (by value), so the
        mode is baked per launch into captured graphs."""
        if self.is_adaptive_lr and self.schedule_type == 'standard':
            self.opt_cfg.adaptive_lr = 3 if (u + 1) % self.num_minibatches == 0 else 2
        elif self.is_adaptive_lr:
            self.opt_cfg.adaptive_lr = 0 if getattr(self, '_hold_sched', False) else 1

    def _build_cfg_structs(self):
        """POD structs passed (by value at launch) to the kernels; baked into captured graphs, so any change
        drops the captured graph."""
        self.loss_cfg = ops.LossCfg(float(self.e_clip), float(self.critic_coef),
                                    float(self.bounds_loss_coef) if self.bounds_loss_coef is not None else 0.0,
                                    int(self.bounds_loss_coef is not None),
                                    {'bound': 1, 'regularisation': 2}.get(self.bound_loss_type, 0), int(bool(self.clip_value)),
                                    int(bool(self.use_smooth_clamp)), int(bool(self.ppo)))
        sched = self.scheduler
        self.opt_cfg = ops.OptCfg(0.9, 0.999, 1e-8, float(self.weight_decay), float(self.grad_norm),
                                  float(getattr(sched, 'kl_threshold', 0.0)), float(getattr(sched, 'min_lr', 1e-6)),
                                  float(getattr(sched, 'max_lr', 1e-2)), float(getattr(sched, 'lr_multiplier', 1.5)),
                                  1.0 / self.world_size, int(bool(self.truncate_grads)),
                                  int(self.is_adaptive_lr))      # 'standard': 2 / 3 per launch (_set_sched_mode)
        rs = self.rewards_shaper
        self.shaper_cfg = ops.ShaperCfg(float(rs.scale_value), float(rs.shift_value), float(rs.min_val), float(rs.max_val),
                                        float(self.gamma), int(bool(rs.log_val)), int(bool(self.value_bootstrap)))
        self._graph_update = None
        self._graph_epoch = None

    # =============================================================================== env plumbing
    def cast_obs(self, obs, name='obs'):
        if isinstance(obs, torch.Tensor):
            self.is_tensor_obses = True
            # the kernels read raw fp32 row-major device memory: anything else (float64 / half observations, a strided view such as
            # obs_buf[:, :D], a tensor on another device) is normalised once here, like the reference's torch ops would accept it
            if obs.dtype != torch.float32 or obs.device != self.device_t or not obs.is_contiguous():
                obs = obs.to(device=self.device_t, dtype=torch.float32).contiguous()
            return obs
        if isinstance(obs, np.ndarray):
            # host env: async H2D on the compute stream.  If the env hands out page-locked memory (e.g. a pinned ring) the DMA
            # reads it directly; otherwise stage through a pinned buffer first.  `name` keys the staging buffers: two views of equal
            # shape (actor obs / critic states) must not share one
            key = (name, obs.shape, obs.dtype.str)
            buf = self._pinned.get(key)
            if buf is None:
                buf = (torch.empty(obs.shape, dtype=torch.float32).pin_memory(),
                       torch.empty(obs.shape, dtype=torch.float32, device=self.device_t))
                self._pinned[key] = buf
            src = torch.from_numpy(obs)
            if src.dtype == torch.float32 and src.is_contiguous() and self._is_pinned(src):
                buf[1].copy_(src, non_blocking=True)
            else:
                buf[0].copy_(src)
                buf[1].copy_(buf[0], non_blocking=True)
            return buf[1]
        return obs

    def _is_pinned(self, t):
        """page-locked check, cached by base address (the driver query costs a few microseconds)"""
        cache = self._pinned.setdefault('_pin_cache', {})
        k = t.data_ptr()
        r = cache.get(k)
        if r is None:
            r = cache[k] = bool(t.is_pinned())
        return r

    def obs_to_tensors(self, obs):
        if isinstance(obs, dict):
            obs = obs['obs'] if 'obs' in obs else obs
        t = self.cast_obs(obs)
        return {'obs': t}

    def env_reset(self):
        obs = self.vec_env.reset()
        obs = self.obs_to_tensors(obs)
        if self.prev_dones is not None:
            self.prev_dones.zero_()
        self._fresh_reset = True            # no pending reset row until the first env step (a2c_common.py:352-353: prev dones = None)
        if getattr(self, 'is_rnn', False) and self.mask_autoreset_rows:
            self._graph_epoch = None        # the captured rollout re-zeroes absorbed states on every step; the first one after a reset must not
        return obs

    def _host_to_dev(self, name, arr, dtype):
        key = (name, arr.shape)
        buf = self._pinned.get(key)
        if buf is None:
            buf = (torch.empty(arr.shape, dtype=dtype).pin_memory(), torch.empty(arr.shape, dtype=dtype, device=self.device_t))
            self._pinned[key] = buf
        buf[0].copy_(torch.from_numpy(np.ascontiguousarray(arr)).to(dtype))
        buf[1].copy_(buf[0], non_blocking=True)
        return buf[1]

    def env_step(self, actions):
        """a2c_common.py:708-719 (+ preprocess_actions :1500-1510 already applied by the policy kernel)."""
        if self.is_tensor_obses:
            obs, rewards, dones, infos = self.vec_env.step(actions)
            if isinstance(rewards, torch.Tensor) and (rewards.dtype != torch.float32 or rewards.device != self.device_t or not rewards.is_contiguous()):
                rewards = rewards.to(device=self.device_t, dtype=torch.float32).contiguous()
            return self.obs_to_tensors(obs), rewards, dones, infos
        key = ('act', tuple(actions.shape))
        hb = self._pinned.get(key)
        if hb is None:
            hb = torch.empty(actions.shape, dtype=torch.float32).pin_memory()
            self._pinned[key] = hb
        hb.copy_(actions, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        obs, rewards, dones, infos = self.vec_env.step(hb.numpy())
        obs_t = self.obs_to_tensors(obs)
        rew = self._host_to_dev('rew', np.asarray(rewards), torch.float32)
        dn = self._host_to_dev('done', np.asarray(dones), torch.uint8)
        if isinstance(infos, dict) and 'time_outs' in infos and not isinstance(infos['time_outs'], torch.Tensor):
            infos = dict(infos)
            infos['time_outs'] = self._host_to_dev('tout', np.asarray(infos['time_outs']), torch.uint8)
        return obs_t, rew, dn, infos

    # =============================================================================== policy forward
    def _trunk(self, x, acts, M, rows_per_chunk=None, chunk_stride=0):
        m = self.model
        # with an LSTM in front the MLP input is h (dense, not normalised)
        nm, ns = (None, None) if (self.is_rnn and m.rnn_before_mlp) else self._norm()
        self._lin_fwd(x, m.W[0], m.b[0], acts[0], m.act_id, rows_per_chunk=rows_per_chunk, chunk_stride=chunk_stride,
                       x_ld=m.mlp_in, norm_mean=nm, norm_std=ns, M=M)
        for i in range(1, len(m.units)):
            self._lin_fwd(acts[i - 1], m.W[i], m.b[i], acts[i], m.act_id, M=M)

    def _repack(self):
        """bf16 operand copy of the weights for the tcgen05 kernels (after every optimiser step / weight load)."""
        if self.use_tc and self._tensors_ready:
            m = self.model
            ops.tc_pack_weights(m.W[0], m.W[1], m.W[2], m.W_head, m.D, m.units, self.actions_num, self.wpack)
        if getattr(self, 'gemm_tc', False) and self._tensors_ready:
            ops.cast_bf16(self.model.flat, self.wbf)

    def _norm(self):
        m = self.model
        return (m.running_mean_std.mean_f32, m.running_mean_std.std_f32) if self.normalize_input else (None, None)

    def _lstm_step(self, obs, h_in, c_in, h_out, c_out):
        """one LSTM step for all N envs (seq_length 1, models.py -> network_builder.py:452-492 -> recurrent.py): returns h_out"""
        m, N = self.model, self.num_actors
        nm, ns = self._norm() if m.rnn_before_mlp else (None, None)      # after the MLP the LSTM reads the trunk output
        self._lin_fwd(obs, m.W_ih, m.b_ih, self.r_gates, 0, x_ld=m.rnn_in, norm_mean=nm, norm_std=ns, M=N)
        self._lin_fwd(h_in, m.W_hh, m.b_hh, self.r_gates, 0, M=N, accumulate=True)
        ops.lstm_cell_fwd(self.r_gates, c_in, c_out, h_out, N, m.rnn_units)
        return h_out

    def _policy_step(self, obs, t, noise=None):
        m, N, A = self.model, self.num_actors, self.actions_num
        if self.use_tc and not self.rollout_fp32:
            nm, ns = self._norm()
            ops.tc_mlp_fwd_rollout(obs, m.D, nm, ns, self.wpack, m.b, m.b_head, m.sigma, m.units, N, A,
                                   m.value_mean_std.running_mean, m.value_mean_std.running_var, self.normalize_value, noise,
                                   self.rng_seed, self.rng_epoch, t, self.actions[t], self.mus[t], self.sigmas[t],
                                   self.neglogpacs[t], self.values[t], self.env_actions, self.clip_actions, self.actions_low,
                                   self.actions_high, self.dones, self.dones_buf[t], self.prev_dones,
                                   None if self.valid is None else self.valid[t], l1_scratch=self.tc_l1_scratch, activation=m.act_id)
            return
        if self.is_rnn and m.rnn_before_mlp:
            obs = self._lstm_step(obs, self.rnn_h, self.rnn_c, self.rnn_h, self.rnn_c)
        self._trunk(obs, self.ra, N)
        a_last = self.ra[-1]
        if self.is_rnn and not m.rnn_before_mlp:
            a_last = self._lstm_step(a_last, self.rnn_h, self.rnn_c, self.rnn_h, self.rnn_c)
        ops.policy_head_sample(a_last, m.W_head, m.b_head, m.logstd_in, m.value_mean_std.running_mean,
                               m.value_mean_std.running_var, self.normalize_value, noise, self.rng_seed, self.rng_epoch, t,
                               self.actions[t], self.mus[t], self.sigmas[t], self.neglogpacs[t], self.values[t],
                               self.env_actions, self.clip_actions, self.actions_low, self.actions_high,
                               self.dones, self.dones_buf[t], self.prev_dones, None if self.valid is None else self.valid[t],
                               N, A)

    def get_values(self, obs):
        """a2c_common.py:603-626"""
        o = obs['obs'] if isinstance(obs, dict) else obs
        m, N, A = self.model, self.num_actors, self.actions_num
        if self.use_tc and not self.rollout_fp32:
            nm, ns = self._norm()
            ops.tc_mlp_fwd_rollout(o, m.D, nm, ns, self.wpack, m.b, m.b_head, m.sigma, m.units, N, A,
                                   m.value_mean_std.running_mean, m.value_mean_std.running_var, self.normalize_value, None, 0, None,
                                   0, None, None, None, None, self.last_values, None, False, None, None, None, None, None, None,
                                   values_only=True, l1_scratch=self.tc_l1_scratch, activation=m.act_id)
            return self.last_values.unsqueeze(1)
        if self.is_rnn and m.rnn_before_mlp:     # get_values does not advance the agent's rnn states (a2c_common.py:603-626)
            o = self._lstm_step(o, self.rnn_h, self.rnn_c, self.r_tmp_h, self.r_tmp_c)
        self._trunk(o, self.ra, N)
        a_last = self.ra[-1]
        if self.is_rnn and not m.rnn_before_mlp:
            a_last = self._lstm_step(a_last, self.rnn_h, self.rnn_c, self.r_tmp_h, self.r_tmp_c)
        ops.policy_head_sample(a_last, m.W_head, m.b_head, m.sigma, m.value_mean_std.running_mean,
                               m.value_mean_std.running_var, self.normalize_value, None, 0, None, 0, None, None, None, None,
                               self.last_values, None, False, None, None, None, None, None, None, N, A, values_only=True)
        return self.last_values.unsqueeze(1)

    def get_action_values(self, obs, noise=None):
        """a2c_common.py:581-601.  Runs the policy on `obs` (writes arena step 0 scratch) and returns the result dict."""
        o = obs['obs'] if isinstance(obs, dict) else obs
        self._policy_step(o, 0, noise)
        return {'actions': self.actions[0], 'neglogpacs': self.neglogpacs[0], 'values': self.values[0].unsqueeze(1),
                'mus': self.mus[0], 'sigmas': self.sigmas[0], 'rnn_states': None}

    # =============================================================================== rollout
    def _rollout(self, noise=None):
        """a2c_common.py:985-1069 without the eager launches: obs copy, trunk, head+sample+store, env, post-step."""
        H, N = self.horizon_length, self.num_actors
        step_time = 0.0
        wants_idx = getattr(self.algo_observer, 'wants_done_indices', True)
        wants_infos = getattr(self.algo_observer, 'wants_infos', False)
        if hasattr(self.vec_env, 'begin_rollout'):
            self.vec_env.begin_rollout()
        self.model.refresh_sigma_floor()          # weights may have been loaded since the last update (no-op unless min_sigma > 0)
        for t in range(H):
            obs = self.obs['obs']
            self.obses[t].copy_(obs)
            if self.is_rnn and t % self.seq_length == 0:      # play_steps_rnn: a2c_common.py:1081-1083
                self.rnn_h0[t // self.seq_length].copy_(self.rnn_h)
                self.rnn_c0[t // self.seq_length].copy_(self.rnn_c)
            self._policy_step(obs, t, None if noise is None else noise[t])
            if self.is_rnn and self.mask_autoreset_rows and not getattr(self, '_fresh_reset', False):
                # a2c_common.py:1097-1106: on a filler reset row (previous step ended the episode; self.dones still holds that step's
                # flags) the forward just absorbed the dead episode's terminal obs into the zeroed state -- zero it again
                ops.rnn_mask_rows(self.rnn_h, N, 0, self.rnn_h, N, self.model.rnn_units, done=self.dones, done_rpc=N)
                ops.rnn_mask_rows(self.rnn_c, N, 0, self.rnn_c, N, self.model.rnn_units, done=self.dones, done_rpc=N)
            self._fresh_reset = False
            t0 = time.perf_counter()
            self.obs, rewards, dones, infos = self.env_step(self.env_actions)
            step_time += time.perf_counter() - t0
            tout = infos.get('time_outs') if (self.value_bootstrap and isinstance(infos, dict)) else None
            ops.post_step(rewards, dones, tout, self.values[t], None if self.valid is None else self.valid[t], self.rewards[t],
                          self.dones, self.prev_dones, self.ep_state, self.meter, self.games_to_track, self.post_scratch,
                          self.counters[0:1], N, self.shaper_cfg)
            if self.is_rnn:     # zero the states of finished episodes (a2c_common.py:1150-1153)
                ops.rnn_mask_rows(self.rnn_h, N, 0, self.rnn_h, N, self.model.rnn_units, done=self.dones, done_rpc=N)
                ops.rnn_mask_rows(self.rnn_c, N, 0, self.rnn_c, N, self.model.rnn_units, done=self.dones, done_rpc=N)
            if wants_idx:
                self.algo_observer.process_infos(infos, self.dones.nonzero(as_tuple=False))
            elif wants_infos:       # observers that read the infos but not the done indices: no host sync
                self.algo_observer.process_infos(infos, None)
        self.get_values(self.obs)
        if hasattr(self.vec_env, 'end_rollout'):
            self.vec_env.end_rollout()
        ops.bump_u64(self.rng_epoch)
        self._meter_cache = None
        return step_time

    def _gae_and_prepare(self):
        if self.is_rnn and self.mask_autoreset_rows:      # train-time state-reset flags (a2c_common.py:1180-1191); GAE uses the plain dones
            ops.rnn_train_dones(self.dones_buf, self.valid, self.rnn_dones_buf)
        nb = ops.gae_fused(self.rewards, self.values, self.dones_buf, self.last_values, self.dones, self.valid, self.advs,
                           self.returns, self.gae_partials, self.gamma, self.tau)
        self._prepare(nb)

    def _prepare(self, n_partials):
        m = self.model
        ops.prepare_batch(self.values, self.returns, self.valid, self.gae_partials, n_partials, m.value_mean_std.running_mean,
                          m.value_mean_std.running_var, m.value_mean_std.count, self.old_values_n, self.returns_n,
                          self.advs_n, self.normalize_value, self.normalize_advantage and not self.normalize_rms_advantage,
                          freeze_stats=bool(self.config.get('freeze_critic', False)))
        if self.normalize_rms_advantage:
            # a2c_common.py:1622-1632: advantages = advantage_mean_std(advantages[, mask]) -- EMA update from the valid rows, then
            # every row normalised with the updated statistics and clamped to +-5
            ops.adv_ema_normalize(self.advs_n, self.gae_partials, n_partials, self.adv_ema_state, self.adv_ema_step,
                                  self.adv_rms_momentum, training=True)
        if self.mask_autoreset_rows:
            ops.mask_inv_counts(self.valid, self.horizon_length, self.num_actors, self.envs_per_mb, self.inv_counts)
        if self.use_mb_moments:
            # obs are fixed for the whole update phase: batch sums of every minibatch in ONE pass over the arena
            ops.obs_mb_moments(self.obses, m.D, self.horizon_length, self.num_actors, self.envs_per_mb,
                               m.running_mean_std.running_mean, self.mbmom, self.mb_shift, self.mom_scratch, self.mb_counters)

    def play_steps(self, noise=None):
        """Public mirror of A2CBase.play_steps: runs the rollout + GAE and returns the reference's batch_dict
        (flat [env*H+t] COPIES of the arena; the fused path never needs them)."""
        self.init_tensors()
        step_time = self._rollout(noise)
        nb = ops.gae_fused(self.rewards, self.values, self.dones_buf, self.last_values, self.dones, self.valid, self.advs,
                           self.returns, self.gae_partials, self.gamma, self.tau)
        self._n_gae_partials = nb
        fl = swap_and_flatten01
        batch_dict = {'actions': fl(self.actions), 'neglogpacs': fl(self.neglogpacs), 'values': fl(self.values.unsqueeze(2)),
                      'mus': fl(self.mus), 'sigmas': fl(self.sigmas), 'obses': fl(self.obses), 'dones': fl(self.dones_buf),
                      'returns': fl(self.returns.unsqueeze(2)), 'played_frames': self.batch_size, 'step_time': step_time}
        if self.mask_autoreset_rows:
            batch_dict['rnn_masks'] = fl(self.valid)
        self._batch_dict_ids = {k: (v.data_ptr(), v._version) for k, v in batch_dict.items() if torch.is_tensor(v)}
        return batch_dict

    def prepare_dataset(self, batch_dict):
        """a2c_common.py:1586-1660.  Accepts the dict from play_steps (possibly edited by the caller: edited or
        foreign tensors are scattered back into the arena first)."""
        H, N = self.horizon_length, self.num_actors
        unfl = lambda t: t.reshape(N, H, *t.shape[1:]).transpose(0, 1)   # noqa: E731
        ids = getattr(self, '_batch_dict_ids', {})
        dirty = False
        for k, dst in (('actions', self.actions), ('neglogpacs', self.neglogpacs), ('values', self.values.unsqueeze(2)),
                       ('mus', self.mus), ('sigmas', self.sigmas), ('obses', self.obses), ('returns', self.returns.unsqueeze(2)),
                       ('rnn_masks', None if self.valid is None else self.valid)):
            v = batch_dict.get(k)
            if v is None or dst is None:
                continue
            if ids.get(k) != (v.data_ptr(), v._version):
                dst.copy_(unfl(v.to(self.device_t)))
                dirty = True
        if dirty or not hasattr(self, '_n_gae_partials'):
            self._n_gae_partials = ops.batch_moments(self.values, self.returns, self.valid, self.gae_partials)
        self._prepare(self._n_gae_partials)
        self.dataset.update_values_dict({'ready': True})

    # =============================================================================== update
    def _minibatch_update(self, i, u):
        """calc_gradients + trancate_gradients_and_step for minibatch i; u = flat update index (stats row)."""
        m, H, N, A = self.model, self.horizon_length, self.num_actors, self.actions_num
        epm, mb = self.envs_per_mb, self.minibatch_size
        e0 = i * epm
        x = self.obses[0, e0:]
        L = len(m.units)
        if self.normalize_input:
            rms = m.running_mean_std
            if self.use_mb_moments:
                if u == 0 or getattr(self, '_compat_mode', False):    # later minibatches are merged by the previous update's optimiser kernel
                    ops.obs_stats_merge(self.mbmom[i], self.mb_shift, m.D, mb, rms.running_mean, rms.running_var, rms.count,
                                        rms.mean_f32, rms.std_f32)
            else:
                ops.moments_update(x, m.D, epm, H, N, rms.running_mean, rms.running_var, rms.count, rms.mean_f32, rms.std_f32,
                                   self.mom_scratch, self.counters[1:2])
        if self.use_tc:
            self._minibatch_update_tc(i, u, x, e0)
            return
        rnn_first = self.is_rnn and m.rnn_before_mlp
        rnn_last = self.is_rnn and not m.rnn_before_mlp
        if rnn_first:
            self._lstm_window_fwd(e0)
            self._trunk(self.t_hmlp, self.ta, mb)
        else:
            self._trunk(x, self.ta, mb, rows_per_chunk=epm, chunk_stride=N)
        if rnn_last:        # MLP -> LSTM -> heads: the heads read the LSTM output and hand back dL/dh (no activation in between)
            self._lstm_window_fwd(e0)
            a_last, d_alast, act_last = self.t_hmlp, self.t_dHmlp, 0
        else:
            a_last, d_alast, act_last = self.ta[-1], self.dA[-1], m.act_id
        nb = ops.ppo_head_loss(a_last, m.W_head, m.b_head, m.logstd_in, self.actions[0, e0:], self.mus[0, e0:],
                               self.sigmas[0, e0:], self.old_values_n[0, e0:], self.returns_n[0, e0:], self.neglogpacs[0, e0:],
                               self.advs_n[0, e0:], None if self.valid is None else self.valid[0, e0:], epm, N, mb, A,
                               self.loss_cfg, None if self.inv_counts is None else self.inv_counts[i:i + 1], self.d_head,
                               d_alast, act_last, self.loss_partials)
        gv = self._gv[u & 1]
        ops.ppo_loss_finalize(self.loss_partials, nb, A, self.entropy_coef_dev, self.stats[u], gv['g_sigma'], gv['kl'])
        if m.min_sigma > 0:      # the kernels differentiated with respect to log(exp(raw) + min_sigma): chain to the raw parameter
            gv['g_sigma'].mul_(m.sigma_chain)
        P = m.num_params
        # row splits of the head / MLP weight gradients.  A recurrent policy's partial arena has seq_length x n_splits rows (one group per
        # BPTT step, _lstm_window_bwd); the layers outside the window may spread over all of them: more CTAs per GEMM, same reduction
        S = min(self.part_rows, max(self.n_splits, mb // 256)) if self.gemm_tc else self.n_splits
        off_wh, _ = m.layout['W_head']
        off_bh, _ = m.layout['b_head']
        self._lin_bww(self.d_head, a_last, self.part[0, off_wh:], self.part[0, off_bh:], m.Hl, A + 1, S, M=mb,
                              split_stride=P)
        if rnn_last:
            self._lstm_window_bwd(e0)       # also fills dA[-1] = dL/d(pre-activation of the last MLP layer)
        nm = m.running_mean_std.mean_f32 if self.normalize_input else None
        ns = m.running_mean_std.std_f32 if self.normalize_input else None
        for l in range(L - 1, -1, -1):
            off_w, shp = m.layout[f'W{l}']
            off_b, _ = m.layout[f'b{l}']
            if l > 0:
                self._lin_bww(self.dA[l], self.ta[l - 1], self.part[0, off_w:], self.part[0, off_b:], shp[1], shp[0], S,
                                      M=mb, split_stride=P)
                self._lin_bwd(self.dA[l], m.W[l], self.ta[l - 1], self.dA[l - 1], m.act_id, M=mb)
            elif rnn_first:
                self._lin_bww(self.dA[0], self.t_hmlp, self.part[0, off_w:], self.part[0, off_b:], shp[1], shp[0], S, M=mb,
                                      split_stride=P)
                self._lin_bwd(self.dA[0], m.W[0], None, self.t_dHmlp, 0, M=mb)
                self._lstm_window_bwd(e0)
            else:
                self._lin_bww(self.dA[0], x, self.part[0, off_w:], self.part[0, off_b:], shp[1], shp[0], S,
                                      rows_per_chunk=epm, chunk_stride=N, x_ld=m.D, norm_mean=nm, norm_std=ns, M=mb,
                                      split_stride=P)
        ops.reduce_splits(self.part[0, A:], gv['grad'][A:], P - A, self.part_rows, split_stride=P)
        if m.grad_mask is not None:      # separate trunks: the structural zeros of the block layout get no gradient (model.py)
            gv['grad'][:P].mul_(m.grad_mask)
        self._step_optimizer(u, gv, P)
        m.refresh_sigma_floor()          # no-op unless min_sigma > 0

    def _lstm_window_fwd(self, e0):
        """Training forward of the LSTM over the seq_length window of every sequence of the minibatch (network_builder.py:452-492,
        recurrent.py:26-58): sequences (j, env) in order j*epm + (env - e0); step t uses arena rows (j*T + t, env)."""
        m, H, N, T = self.model, self.horizon_length, self.num_actors, self.seq_length
        epm, Hd = self.envs_per_mb, m.rnn_units
        S = epm * H // T
        nm, ns = self._norm() if m.rnn_before_mlp else (None, None)
        # window-initial states = snapshots taken during the rollout, zeroed where the episode ended entering step 0
        dn = self.rnn_dones_buf if self.rnn_dones_buf is not None else self.dones_buf
        ops.rnn_mask_rows(self.rnn_h0[0, e0:], epm, N, self.t_hin[0], S, Hd, done=dn[0, e0:], done_rpc=epm, done_stride=T * N)
        ops.rnn_mask_rows(self.rnn_c0[0, e0:], epm, N, self.t_cin[0], S, Hd, done=dn[0, e0:], done_rpc=epm, done_stride=T * N)
        for t in range(T):
            # step-t inputs of all S sequences: arena observations (LSTM first) or the trunk output rows (j*T + t)*epm + e (LSTM last)
            xin, xstride = (self.obses[t, e0:], T * N) if m.rnn_before_mlp else (self.ta[-1][t * epm:], T * epm)
            self._lin_fwd(xin, m.W_ih, m.b_ih, self.t_gates[t], 0, rows_per_chunk=epm, chunk_stride=xstride, x_ld=m.rnn_in,
                           norm_mean=nm, norm_std=ns, M=S)
            self._lin_fwd(self.t_hin[t], m.W_hh, m.b_hh, self.t_gates[t], 0, M=S, accumulate=True)
            last = t == T - 1
            ops.lstm_cell_fwd(self.t_gates[t], self.t_cin[t], self.t_c[t], self.t_hdense, S, Hd,
                              h_scatter=self.t_hmlp[t * epm:], scatter_rpc=epm, scatter_stride=T * epm,
                              hin_next=None if last else self.t_hin[t + 1], cin_next=None if last else self.t_cin[t + 1],
                              done_next=None if last else dn[t + 1, e0:], done_rpc=epm, done_stride=T * N)

    def _lstm_window_bwd(self, e0):
        """BPTT over the window: cell backward, weight gradients of W_ih / W_hh (+ both biases) per step into their own split rows,
        dgrad through W_hh to the previous step."""
        m, H, N, T = self.model, self.horizon_length, self.num_actors, self.seq_length
        epm, Hd, P, Ssp = self.envs_per_mb, m.rnn_units, m.num_params, self.n_splits
        S = epm * H // T
        nm, ns = self._norm() if m.rnn_before_mlp else (None, None)
        o_wih, o_whh, o_bih, o_bhh = (m.layout[k][0] for k in ('W_ih', 'W_hh', 'b_ih', 'b_hh'))
        dn = self.rnn_dones_buf if self.rnn_dones_buf is not None else self.dones_buf
        for t in range(T - 1, -1, -1):
            last = t == T - 1
            ops.lstm_cell_bwd(self.t_gates[t], self.t_c[t], self.t_cin[t], self.t_dgates, self.t_dcin[t & 1], S, Hd,
                              dH=self.t_dHmlp[t * epm:], scatter_rpc=epm, scatter_stride=T * epm,
                              dhin_next=None if last else self.t_dhin, dcin_next=None if last else self.t_dcin[(t + 1) & 1],
                              done_next=None if last else dn[t + 1, e0:], done_rpc=epm, done_stride=T * N)
            row = t * Ssp
            xin, xstride = (self.obses[t, e0:], T * N) if m.rnn_before_mlp else (self.ta[-1][t * epm:], T * epm)
            self._lin_bww(self.t_dgates, xin, self.part[row, o_wih:], self.part[row, o_bih:], m.rnn_in, 4 * Hd, Ssp,
                                  rows_per_chunk=epm, chunk_stride=xstride, x_ld=m.rnn_in, norm_mean=nm, norm_std=ns, M=S, split_stride=P)
            self._lin_bww(self.t_dgates, self.t_hin[t], self.part[row, o_whh:], self.part[row, o_bhh:], Hd, 4 * Hd, Ssp, M=S,
                                  split_stride=P)
            if t > 0:
                self._lin_bwd(self.t_dgates, m.W_hh, None, self.t_dhin, 0, M=S)
            if not m.rnn_before_mlp:
                # dgrad through W_ih into the trunk: sequences j*epm..(j+1)*epm-1 at step t are trunk rows (j*T + t)*epm.., one dense
                # epm-row block each; the last MLP layer's activation derivative is folded in (dA[-1] is d pre-activation)
                for j in range(H // T):
                    r0 = (j * T + t) * epm
                    self._lin_bwd(self.t_dgates[j * epm:], m.W_ih, self.ta[-1][r0:], self.dA[-1][r0:], m.act_id, M=epm)

    def _minibatch_update_tc(self, i, u, x, e0):
        """bf16 tcgen05 edition: fused fwd+loss kernel, two backward kernels, split reduce, Adam, repack."""
        m, H, N, A = self.model, self.horizon_length, self.num_actors, self.actions_num
        epm, mb, P = self.envs_per_mb, self.minibatch_size, self.model.num_params
        nm, ns = self._norm()
        nb = ops.tc_mlp_fwd_train(x, epm, N, m.D, nm, ns, self.wpack, m.b, m.b_head, m.sigma, m.units, mb, A, self.actions[0, e0:],
                                  self.mus[0, e0:], self.sigmas[0, e0:], self.old_values_n[0, e0:], self.returns_n[0, e0:],
                                  self.neglogpacs[0, e0:], self.advs_n[0, e0:], None if self.valid is None else self.valid[0, e0:],
                                  self.loss_cfg, None if self.inv_counts is None else self.inv_counts[i:i + 1], self.tc_act,
                                  self.tc_dhead, self.loss_partials, xtile=self.tc_xt, activation=m.act_id)
        npart = ops.tc_mlp_bwd(x, epm, N, m.D, nm, ns, self.wpack, m.units, mb, A, self.tc_act, self.tc_dhead, self.tc_delta2,
                               self.tc_delta1, self.part, self.part.shape[1], self.tc_offs, xtile=self.tc_xt, activation=m.act_id,
                               pipelined_wgrad=self.tc_pipelined_wgrad)
        gv = self._gv[u & 1]
        self._set_sched_mode(u)
        if not self.multi_gpu:
            # no exchange between the reduction and the optimiser: one fused launch (reduce + finalise + clip + Adam + repack)
            ops.reduce_adam(self.part, npart, self.part.shape[1], self.loss_partials, nb, A, self.entropy_coef_dev, self.stats[u], gv['kl'], gv['grad'],
                            m.flat, m.exp_avg, m.exp_avg_sq, P, self.opt_state, self.opt_cfg, self.counters[2:3], self.ra_nrm, self.ra_bar,
                            wpack=self.wpack, pack_table=self.pack_table, merge_next=self._merge_next(u))
            return
        if self.fused_allreduce and self.fused_split_allreduce:
            ops.reduce_allreduce_adam(self.part, npart, self.part.shape[1], self.loss_partials, nb, A, self.entropy_coef_dev, self.stats[u],
                                      self.peer_table, u & 1, self.global_rank, self.my_cta_flags_ptr, self.ar_seq, self.ar_red, m.flat,
                                      m.exp_avg, m.exp_avg_sq, P, self.opt_state, self.opt_cfg, self.counters[2:3], self.ra_nrm,
                                      self.ra_bar, wpack=self.wpack, pack_table=self.pack_table, merge_next=self._merge_next(u))
            return
        ops.reduce_finalize(self.part[0, A:], gv['grad'][A:], P - A, npart, self.part.shape[1], self.loss_partials, nb, A, self.entropy_coef_dev,
                            self.stats[u], gv['g_sigma'], gv['kl'])
        self._step_optimizer(u, gv, P, wpack=self.wpack, pack_table=self.pack_table)

    def _update_all(self):
        u = 0
        if self.is_adaptive_lr and self.schedule_type == 'standard':
            self.opt_state[4:6].zero_()      # a mini-epoch's KL accumulators never survive an interrupted epoch
        resume_lr = getattr(self, '_resume_opt_lr', None)
        self._resume_opt_lr = None
        for _ in range(self.mini_epochs_num):
            for i in range(self.num_minibatches):
                if u == 0 and resume_lr is not None and self.is_adaptive_lr:
                    # the restored optimizer lr drives this one step; the scheduler step that follows it starts from last_lr
                    if self.schedule_type != 'per_minibatch':
                        raise NotImplementedError("resume with schedule_type 'standard'")
                    self._hold_sched = True
                self._minibatch_update(i, u)
                if u == 0 and resume_lr is not None and self.is_adaptive_lr:
                    self._hold_sched = False
                    self.opt_cfg.adaptive_lr = 1
                    kl, scale = self._kl_for_sched(0)
                    ops.lr_schedule_apply(self.opt_state, kl, scale, self.last_lr, self.opt_cfg)
                elif u == 0 and (self._sched_switch or resume_lr is not None):
                    self.opt_state[0:1].copy_(self.lr_next_dev)
                    self.entropy_coef_dev.copy_(self.ent_next_dev)
                u += 1

    def _kl_for_sched(self, u):
        """device location and scale of the KL the scheduler saw for update u (rank mean on several GPUs)"""
        if self.fused_allreduce:
            return self.ar_red[self.model.num_params:], 1.0 / self.world_size
        if self.multi_gpu:
            return self._gv[u & 1]['kl'], 1.0 / self.world_size
        return self.stats[u][4:5], 1.0

    def _run_update(self):
        """Eager the first time (module loading, attribute setup); from the second epoch on the whole
        mini_epochs x num_minibatches sequence replays as ONE CUDA graph (capture executes nothing)."""
        if not self.use_cuda_graph or (self.multi_gpu and not self.graph_multi_gpu):
            self._update_all()
            return
        if not getattr(self, '_update_warm', False):
            self._update_all()
            self._update_warm = True
            return
        if self._graph_update is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._update_all()
            self._graph_update = g
        self._graph_update.replay()

    # =============================================================================== reference-style per-minibatch API
    def train_actor_critic(self, input_dict, opt_step=True):
        """a2c_continuous.py:236-239.  `input_dict` must come from ``self.dataset[i]``."""
        i = input_dict.get('_mb_index')
        if i is None:
            raise NotImplementedError('train_actor_critic needs a minibatch produced by agent.dataset[i]')
        self.init_tensors()
        u = self._compat_u = getattr(self, '_compat_u', -1) + 1
        u %= self.n_updates
        self._compat_mode = True     # caller-driven order: merge the obs statistics per call, not in the optimiser tail
        try:
            self._minibatch_update(i, u)
        finally:
            self._compat_mode = False
        st = self.stats[u]
        e0, e1 = i * self.envs_per_mb, (i + 1) * self.envs_per_mb
        self.train_result = (st[0], st[1], st[2], st[4], self.last_lr, 1.0, swap_and_flatten01(self.mus[:, e0:e1]),
                             swap_and_flatten01(self.sigmas[:, e0:e1]), st[3])
        return self.train_result

    def calc_gradients(self, input_dict):
        return self.train_actor_critic(input_dict)

    # =============================================================================== epoch
    def set_eval(self):
        self.model.eval()

    def set_train(self):
        self.model.train()

    def train_epoch(self, noise=None):
        """a2c_common.py:1517-1584.  Returns the reference tuple; the per-minibatch scalars are 0-dim views of
        one device stats block, read back with ONE D2H copy + sync per epoch."""
        self.init_tensors()
        if self.vec_env is not None and hasattr(self.vec_env, 'set_train_info'):
            self.vec_env.set_train_info(self.frame, self)
        ev = self._events
        self.set_eval()
        if self._lr_dirty():
            self.opt_state[0:1].fill_(self.last_lr)
        if getattr(self, '_resume_opt_lr', None) is not None:       # first epoch after a restore: one step on the checkpoint's lr
            self.opt_state[0:1].fill_(self._resume_opt_lr)
            if not self._sched_switch:
                self.lr_next_dev.fill_(self.last_lr)
                self.ent_next_dev.fill_(float(self.entropy_coef))
        if self._sched_switch:      # this epoch's schedule value, used from the second minibatch on (outside any captured graph)
            lr_b, ent_b = self.scheduler.update(self.last_lr, self.entropy_coef, self.epoch_num, self.frame, 0.0)
            self.lr_next_dev.fill_(float(lr_b))
            self.ent_next_dev.fill_(float(ent_b))
        whole = noise is None and self._whole_epoch_graph_ok()
        ev[0].record()
        if whole and getattr(self, '_epoch_warm', False):
            # rollout + GAE + prepare + every minibatch update as ONE graph launch (env kernels included)
            if self._graph_epoch is None:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._rollout(None)
                    self._gae_and_prepare()
                    self._update_all()
                    self.sync_running_stats()     # in-place tensor math + one NCCL all-reduce: graph-capturable
                self._graph_epoch = g
            self._graph_epoch.replay()
            self._meter_cache = None
            step_time = 0.0
            ev[1].record()
            split_known = False
        else:
            step_time = self._rollout(noise)
            self._gae_and_prepare()
            ev[1].record()
            self.set_train()
            self._run_update()
            self.sync_running_stats()
            self._epoch_warm = True
            split_known = True
        self.set_train()
        self.curr_frames = self.batch_size
        self.algo_observer.after_steps()
        ev[2].record()
        # one D2H read-back per epoch: stats rows + (lr, step) + meter
        self.host_stats.copy_(self.stats, non_blocking=True)
        self.host_state[0:2].copy_(self.opt_state[0:2], non_blocking=True)
        self.host_state[2:10].copy_(self.meter, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self._meter_cache = self.host_state[2:10].numpy().copy()
        st = self.host_stats.clone()
        hs, n = self.host_state, 0
        new_lr = float(hs[n])
        if not self.is_adaptive_lr:
            # linear / identity schedules depend only on (epoch, frame): evaluate on the host once per epoch
            # (the reference re-evaluates the same value after every minibatch, a2c_common.py:1557-1563)
            new_lr, self.entropy_coef = self.scheduler.update(self.last_lr, self.entropy_coef, self.epoch_num, self.frame,
                                                              float(st[:, 4].mean()))
            self.entropy_coef_dev.fill_(float(self.entropy_coef))
        self.last_lr = new_lr
        self._lr_synced = new_lr
        if split_known:
            play_time = ev[0].elapsed_time(ev[1]) * 1e-3
            update_time = ev[1].elapsed_time(ev[2]) * 1e-3
            self._play_frac = play_time / max(play_time + update_time, 1e-12)
        else:   # whole-epoch graph: one launch, split by the ratio measured on the last eager epoch
            tot = ev[0].elapsed_time(ev[2]) * 1e-3
            play_time = tot * getattr(self, '_play_frac', 0.15)
            update_time = tot - play_time
        total_time = play_time + update_time
        a_losses = [st[u, 0] for u in range(self.n_updates)]
        c_losses = [st[u, 1] for u in range(self.n_updates)]
        entropies = [st[u, 2] for u in range(self.n_updates)]
        b_losses = [st[u, 3] for u in range(self.n_updates)] if self.bounds_loss_coef is not None else []
        nmb = self.num_minibatches
        kls = [st[e * nmb:(e + 1) * nmb, 4].mean() for e in range(self.mini_epochs_num)]
        self.last_stats = st
        # the tuple's last_lr is what train_actor_critic returned for the LAST minibatch (a2c_common.py:1548, :1582): the lr that
        # minibatch ran on (stats column 7, written by the optimiser kernel), not self.last_lr after the final scheduler step
        return step_time, play_time, update_time, total_time, a_losses, c_losses, b_losses, entropies, kls, float(st[-1, 7]), 1.0

    def _whole_epoch_graph_ok(self):
        """The env step is part of the captured graph only if the env says its step is a pure stream-ordered sequence on
        static buffers (`cuda_graph_capturable`), and nothing in the rollout needs the host (done indices for observers)."""
        return (self.use_cuda_graph and self.config.get('b200_cuda_graph_rollout', True) and self.is_tensor_obses
                and getattr(self.vec_env, 'cuda_graph_capturable', False)
                and not getattr(self.algo_observer, 'wants_done_indices', True)
                and not getattr(self.algo_observer, 'wants_infos', False)
                and (not self.multi_gpu or self.graph_multi_gpu))

    def _lr_dirty(self):
        return getattr(self, '_lr_synced', None) != self.last_lr

    # =============================================================================== train loop / checkpoints (agent_base.A2CBase)
    def _on_train_start(self):
        self.curr_frames = self.batch_size_envs

    def _broadcast_weights(self):
        super()._broadcast_weights()
        self._repack()

    def write_stats(self, total_time, epoch_num, step_time, play_time, update_time, a_losses, c_losses, entropies, kls,
                    last_lr, lr_mul, frame, scaled_time, scaled_play_time, curr_frames):
        super().write_stats(total_time, epoch_num, step_time, play_time, update_time, a_losses, c_losses, entropies, kls,
                            last_lr, lr_mul, frame, scaled_time, scaled_play_time, curr_frames)
        if self.bounds_loss_coef is not None:        # a2c_common.py:1705-1706 (after write_stats and the observer's scalars)
            self.writer.add_scalar('losses/bounds_loss', float(self.last_stats[:, 3].mean()), frame)

    def set_weights(self, weights):
        super().set_weights(weights)
        self._repack()

    def _optimizer_lr(self):
        # the optimizer's own lr: last_lr, except between a restore and the first step after it (see _restore_optimizer)
        return self._resume_opt_lr if getattr(self, '_resume_opt_lr', None) is not None else self.last_lr

    def _restore_optimizer(self, lr, step):
        # the first optimiser step after a restore runs on the checkpoint's lr, then update_lr() overwrites it with the scheduler's value
        # computed from this agent's own last_lr (which a restore leaves alone): the checkpoint lr is held for one step (_update_all)
        self._resume_opt_lr = float(lr) if lr is not None else None
        self._graph_update = self._graph_epoch = None
        self._update_warm = self._epoch_warm = False
        self.opt_state.copy_(adam_opt_state(self.last_lr, step, slots=8))
        self._lr_synced = self.last_lr

    def get_full_state_weights(self):
        state = super().get_full_state_weights()
        if self.normalize_rms_advantage:      # a2c_common.py:896-897: GeneralizedMovingStats.state_dict() keys
            st = self.adv_ema_state.cpu()
            state['advantage_mean_std'] = {'step': self.adv_ema_step.cpu().clone(), 'mean': st[0:1].clone(), 'sqrs': st[1:2].clone()}
        return state

    def set_full_state_weights(self, weights, set_epoch=True):
        super().set_full_state_weights(weights, set_epoch=set_epoch)
        if self.normalize_rms_advantage and 'advantage_mean_std' in weights:      # a2c_common.py:909-911
            ams = weights['advantage_mean_std']
            self.adv_ema_state.copy_(torch.cat([ams['mean'].reshape(1).float(), ams['sqrs'].reshape(1).float()]))
            self.adv_ema_step.copy_(ams['step'].reshape(1).to(torch.int32))

    def restore_central_value_function(self, fn):
        # the reference's Runner refuses this before it gets here (torch_runner.py:45-46)
        raise ValueError('Loading critic only works only for asymmetric actor critic')

    def get_param(self, param_name):
        if param_name in ['grad_norm', 'critic_coef', 'bounds_loss_coef', 'entropy_coef', 'kl_threshold', 'gamma', 'tau',
                          'mini_epochs_num', 'e_clip']:
            return getattr(self, param_name)
        elif param_name == 'learning_rate':
            return self.last_lr
        raise NotImplementedError(f"Can't get param {param_name}")

    def set_param(self, param_name, param_value):
        if param_name in ['grad_norm', 'critic_coef', 'bounds_loss_coef', 'entropy_coef', 'gamma', 'tau', 'mini_epochs_num',
                          'e_clip']:
            setattr(self, param_name, param_value)
            self._refresh_cfg()
        elif param_name == 'learning_rate':
            if self.is_adaptive_lr:
                raise NotImplementedError("Can't directly mutate LR on this schedule")
            self.last_lr = float(param_value)
        elif param_name == 'kl_threshold':
            if not self.is_adaptive_lr:
                raise NotImplementedError("Can't directly mutate kl threshold")
            self.kl_threshold = param_value
            self.scheduler.kl_threshold = param_value
            self._refresh_cfg()
        else:
            raise NotImplementedError(f'No param found for {param_value}')

    def _refresh_cfg(self):
        if self._tensors_ready:
            self._build_cfg_structs()
            # the kernels read the entropy coefficient from device memory (graph replays see the new value): keep it in step with a
            # set_param('entropy_coef', v), like the reference, which applies a PBT mutation on the next minibatch
            self.entropy_coef_dev.fill_(float(self.entropy_coef))
            self.ent_next_dev.fill_(float(self.entropy_coef))
            if self.mini_epochs_num * self.num_minibatches != self.n_updates:
                self._resize_updates()

    def _resize_updates(self):
        """set_param('mini_epochs_num', k) after init: everything sized by the number of updates per epoch follows"""
        self.n_updates = self.mini_epochs_num * self.num_minibatches
        self.stats = torch.zeros(self.n_updates, 16, dtype=torch.float32, device=self.device_t)
        self.host_stats = torch.zeros(self.n_updates, 16, dtype=torch.float32).pin_memory()
        self._graph_update = self._graph_epoch = None
        if self.fused_allreduce and self.n_updates % 2 != 0:
            raise NotImplementedError('the fused peer all-reduce alternates exchange buffers by update parity: mini_epochs x '
                                      'num_minibatches must stay even (or set b200_fused_allreduce: False)')
