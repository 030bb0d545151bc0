"""Tensor-level wrappers over the C ABI (include/b200rl.h).  PyTorch is plumbing only: it owns device
memory and the CUDA stream; every op below is one (or two) hand-written sm_100a kernel launches.

There is no CPU path: tensors must live on a CUDA device, and a missing libb200rl.so raises.
"""
import ctypes

import torch

from ._lib import lib, check, ptr, B200RLError

ACT = {'None': 0, None: 0, 'none': 0, 'elu': 1, 'relu': 2, 'tanh': 3}


class LossCfg(ctypes.Structure):
    _fields_ = [('e_clip', ctypes.c_float), ('critic_coef', ctypes.c_float), ('bounds_loss_coef', ctypes.c_float),
                ('has_bounds_loss', ctypes.c_int), ('bound_loss_type', ctypes.c_int), ('clip_value', ctypes.c_int),
                ('use_smooth_clamp', ctypes.c_int), ('ppo', ctypes.c_int)]


class OptCfg(ctypes.Structure):
    _fields_ = [('beta1', ctypes.c_double), ('beta2', ctypes.c_double), ('eps', ctypes.c_double),
                ('weight_decay', ctypes.c_double), ('grad_norm', ctypes.c_double), ('kl_threshold', ctypes.c_double),
                ('min_lr', ctypes.c_double), ('max_lr', ctypes.c_double), ('lr_multiplier', ctypes.c_double),
                ('grad_scale', ctypes.c_double), ('truncate_grads', ctypes.c_int), ('adaptive_lr', ctypes.c_int)]


class ShaperCfg(ctypes.Structure):
    _fields_ = [('scale_value', ctypes.c_float), ('shift_value', ctypes.c_float), ('min_val', ctypes.c_float),
                ('max_val', ctypes.c_float), ('gamma', ctypes.c_float), ('log_val', ctypes.c_int),
                ('value_bootstrap', ctypes.c_int)]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError('rl_games_b200 ops need CUDA tensors (no CPU fallback)')


def compute_gae(mb_rewards, mb_values, mb_dones, last_values, last_dones, gamma, tau, returns_out=None):
    """Drop-in for rl_games.triton_kernels.compute_gae (gae_kernel.py:124-146): same signature, accepts
    non-contiguous views and float or uint8 dones; returns a new [H,N,V] fp32 tensor."""
    _need_cuda(mb_rewards, mb_values, mb_dones, last_values, last_dones)
    H, N, V = mb_rewards.shape
    if mb_rewards.dtype != torch.float32:
        mb_rewards = mb_rewards.float()
    if mb_values.dtype != torch.float32:
        mb_values = mb_values.float()

    def _dn(d):
        if d.dtype in (torch.uint8, torch.bool):
            return d.view(torch.uint8) if d.dtype == torch.bool else d, 1
        return (d if d.dtype == torch.float32 else d.float()), 0
    mb_dones, d_u8 = _dn(mb_dones)
    last_dones, ld_u8 = _dn(last_dones)
    last_values = last_values.contiguous().float()
    last_dones = last_dones.contiguous()
    advs = torch.empty((H, N, V), dtype=torch.float32, device=mb_rewards.device)
    if returns_out is not None:
        assert returns_out.shape == advs.shape and returns_out.is_contiguous()
    rs, vs, ds, as_ = mb_rewards.stride(), mb_values.stride(), mb_dones.stride(), advs.stride()
    check(lib.b200rl_gae_f32(ptr(mb_rewards), ptr(mb_values), ptr(mb_dones), d_u8, ptr(last_values), ptr(last_dones),
                             ld_u8, ptr(advs), ptr(returns_out), H, N, V, rs[0], rs[1], rs[2], vs[0], vs[1], vs[2],
                             ds[0], ds[1], as_[0], as_[1], as_[2], float(gamma), float(tau), _stream()), 'gae')
    return advs


def gae_set_tma(enable):
    """A/B switch: TMA-staged GAE kernel (default) vs the register-chunk kernel; returns the previous setting"""
    return bool(lib.b200rl_gae_set_tma(1 if enable else 0))


def gae_fused(rewards, values, dones_u8, last_values, last_dones_u8, mask, advs, returns, partials, gamma, tau):
    """Fused GAE + returns + moment partials on contiguous [H,N] tensors.  Returns number of partial rows."""
    H, N = rewards.shape
    nb = ctypes.c_int(0)
    check(lib.b200rl_gae_fused_f32(ptr(rewards), ptr(values), ptr(dones_u8), ptr(last_values), ptr(last_dones_u8),
                                   ptr(mask), ptr(advs), ptr(returns), ptr(partials),
                                   0 if partials is None else partials.shape[0], H, N, float(gamma), float(tau),
                                   ctypes.addressof(nb), _stream()), 'gae_fused')
    return nb.value


def prepare_batch(values, returns, mask, partials, n_partials, vms_mean, vms_var, vms_count, old_values_n,
                  returns_n, advs_n, normalize_value, normalize_advantage, freeze_stats=False):
    check(lib.b200rl_prepare_batch_f32(ptr(values), ptr(returns), ptr(mask), ptr(partials), n_partials,
                                       ptr(vms_mean), ptr(vms_var), ptr(vms_count), ptr(old_values_n), ptr(returns_n),
                                       ptr(advs_n), values.numel(), int(normalize_value), int(normalize_advantage),
                                       int(freeze_stats), _stream()), 'prepare_batch')


def adv_ema_normalize(advs, partials, n_partials, ema_state, ema_step, decay, training=True):
    check(lib.b200rl_adv_ema_normalize_f32(ptr(advs), advs.numel(), ptr(partials), n_partials, ptr(ema_state), ptr(ema_step),
                                           float(decay), int(training), _stream()), 'adv_ema_normalize')


def batch_moments(values, returns, mask, partials):
    nb = ctypes.c_int(0)
    check(lib.b200rl_batch_moments_f64(ptr(values), ptr(returns), ptr(mask), ptr(partials), partials.shape[0],
                                       values.numel(), ctypes.addressof(nb), _stream()), 'batch_moments')
    return nb.value


def moments_update(x, D, rows_per_chunk, n_chunks, chunk_stride, mean, var, count, mean_f32, std_f32, scratch, counter,
                   eps=1e-5):
    check(lib.b200rl_moments_update_f64(ptr(x), D, rows_per_chunk, n_chunks, chunk_stride, ptr(mean), ptr(var),
                                        ptr(count), ptr(mean_f32), ptr(std_f32), eps, ptr(scratch),
                                        scratch.numel() // (2 * D), ptr(counter), _stream()), 'moments_update')


def obs_mb_moments(x, D, H, N, envs_per_mb, run_mean, mbmom, mb_shift, scratch, counters):
    check(lib.b200rl_obs_mb_moments_f64(ptr(x), D, H, N, envs_per_mb, ptr(run_mean), ptr(mbmom), ptr(mb_shift), ptr(scratch),
                                        scratch.numel() // (2 * D), ptr(counters), _stream()), 'obs_mb_moments')


def obs_stats_merge(mbmom_i, mb_shift, D, n_rows, mean, var, count, mean_f32, std_f32, eps=1e-5):
    check(lib.b200rl_obs_stats_merge_f64(ptr(mbmom_i), ptr(mb_shift), D, n_rows, ptr(mean), ptr(var), ptr(count), ptr(mean_f32),
                                         ptr(std_f32), eps, _stream()), 'obs_stats_merge')


def refresh_norm(mean, var, mean_f32, std_f32, eps=1e-5):
    check(lib.b200rl_refresh_norm_f32(ptr(mean), ptr(var), ptr(mean_f32), ptr(std_f32), eps, mean.numel(), _stream()),
          'refresh_norm')


def normalize(x, mean, var, denorm=False, eps=1e-5, out=None):
    x = x.contiguous()
    D = mean.numel()
    y = torch.empty_like(x) if out is None else out
    check(lib.b200rl_normalize_f32(ptr(x), ptr(y), ptr(mean), ptr(var), eps, x.numel() // D, D, int(denorm), _stream()),
          'normalize')
    return y


def linear_fwd(X, W, b, Y, act, rows_per_chunk=None, chunk_stride=0, x_ld=None, norm_mean=None, norm_std=None, M=None,
               accumulate=False):
    Nout, K = W.shape
    M = Y.shape[0] if M is None else M
    check(lib.b200rl_linear_fwd_f32(ptr(X), M if rows_per_chunk is None else rows_per_chunk, chunk_stride,
                                    K if x_ld is None else x_ld, ptr(norm_mean), ptr(norm_std), ptr(W), ptr(b), ptr(Y),
                                    M, K, Nout, act, int(accumulate), _stream()), 'linear_fwd')


def linear_bwd_data(dY, W, A_prev, dX, act_prev, M=None):
    Nout, K = W.shape
    M = dY.shape[0] if M is None else M
    check(lib.b200rl_linear_bwd_data_f32(ptr(dY), ptr(W), ptr(A_prev), ptr(dX), M, K, Nout, act_prev, _stream()),
          'linear_bwd_data')


def linear_bwd_weight(dY, X, dW_part, db_part, K, Nout, n_splits, rows_per_chunk=None, chunk_stride=0, x_ld=None,
                      norm_mean=None, norm_std=None, M=None, split_stride=None):
    M = dY.shape[0] if M is None else M
    if split_stride is None:
        assert dW_part.stride(0) == db_part.stride(0) or db_part is None or dW_part.dim() == 3
        split_stride = dW_part.stride(0)
    check(lib.b200rl_linear_bwd_weight_f32(ptr(dY), ptr(X), M if rows_per_chunk is None else rows_per_chunk,
                                           chunk_stride, K if x_ld is None else x_ld, ptr(norm_mean), ptr(norm_std),
                                           ptr(dW_part), ptr(db_part), split_stride, M, K, Nout, n_splits, _stream()),
          'linear_bwd_weight')


def cast_bf16(src, dst):
    """bf16 copy of an fp32 arena (same offsets): the weight operand of the layer-wise tensor-core GEMMs, refreshed once per optimiser step"""
    check(lib.b200rl_cast_bf16(ptr(src), ptr(dst), src.numel(), _stream()), 'cast_bf16')


def _bf16_view_ptr(W, bf16_arena):
    """address of W's twin inside the bf16 copy of the arena W is a view of (bf16_arena = (fp32 arena, bf16 arena)), or None"""
    if bf16_arena is None:
        return None
    flat, fb = bf16_arena
    off = W.data_ptr() - flat.data_ptr()
    if 0 <= off < flat.numel() * 4 and W.is_contiguous():
        return fb.data_ptr() + off // 2
    return None


def linear_fwd_tc(X, W, b, Y, act, rows_per_chunk=None, chunk_stride=0, x_ld=None, norm_mean=None, norm_std=None, M=None,
                  accumulate=False, bf16_arena=None):
    """linear_fwd on the tensor cores (bf16 operands, fp32 accumulate), any layer width"""
    Nout, K = W.shape
    M = Y.shape[0] if M is None else M
    check(lib.b200rl_linear_fwd_tc(ptr(X), M if rows_per_chunk is None else rows_per_chunk, chunk_stride,
                                   K if x_ld is None else x_ld, ptr(norm_mean), ptr(norm_std), ptr(W), _bf16_view_ptr(W, bf16_arena), ptr(b), ptr(Y),
                                   M, K, Nout, act, int(accumulate), _stream()), 'linear_fwd_tc')


def linear_bwd_data_tc(dY, W, A_prev, dX, act_prev, M=None, bf16_arena=None):
    Nout, K = W.shape
    M = dY.shape[0] if M is None else M
    check(lib.b200rl_linear_bwd_data_tc(ptr(dY), ptr(W), _bf16_view_ptr(W, bf16_arena), ptr(A_prev), ptr(dX), M, K, Nout, act_prev, _stream()),
          'linear_bwd_data_tc')


def linear_bwd_weight_tc(dY, X, dW_part, db_part, K, Nout, n_splits, rows_per_chunk=None, chunk_stride=0, x_ld=None,
                         norm_mean=None, norm_std=None, M=None, split_stride=None):
    M = dY.shape[0] if M is None else M
    if split_stride is None:
        split_stride = dW_part.stride(0)
    check(lib.b200rl_linear_bwd_weight_tc(ptr(dY), ptr(X), M if rows_per_chunk is None else rows_per_chunk,
                                          chunk_stride, K if x_ld is None else x_ld, ptr(norm_mean), ptr(norm_std),
                                          ptr(dW_part), ptr(db_part), split_stride, M, K, Nout, n_splits, _stream()),
          'linear_bwd_weight_tc')


def reduce_splits(part, out, n, n_splits, split_stride=None):
    check(lib.b200rl_reduce_splits_f32(ptr(part), ptr(out), n, n_splits, n if split_stride is None else split_stride,
                                       _stream()), 'reduce_splits')


def loss_partial_stride():
    return lib.b200rl_loss_partial_stride()


def ppo_head_loss(a_last, W_head, b_head, logstd, actions, old_mu, old_sigma, old_values_n, returns_n, old_neglogp,
                  advs_n, mask, rows_per_chunk, chunk_stride, M, A, cfg, inv_count, d_head, d_alast, act_last, partials,
                  mu_out=None, value_out=None, neglogp_out=None):
    nb = ctypes.c_int(0)
    Hl = W_head.shape[1]
    check(lib.b200rl_ppo_head_loss_f32(ptr(a_last), Hl, ptr(W_head), ptr(b_head), ptr(logstd), ptr(actions), ptr(old_mu),
                                       ptr(old_sigma), ptr(old_values_n), ptr(returns_n), ptr(old_neglogp), ptr(advs_n),
                                       ptr(mask), rows_per_chunk, chunk_stride, M, A, ctypes.addressof(cfg),
                                       ptr(inv_count), ptr(d_head), ptr(d_alast), act_last, ptr(mu_out), ptr(value_out),
                                       ptr(neglogp_out), ptr(partials), partials.shape[0], ctypes.addressof(nb),
                                       _stream()), 'ppo_head_loss')
    return nb.value


def ppo_loss_finalize(partials, n_partials, A, entropy_coef_dev, stats, d_logstd, kl_out=None):
    check(lib.b200rl_ppo_loss_finalize(ptr(partials), n_partials, A, ptr(entropy_coef_dev), ptr(stats), ptr(d_logstd),
                                       ptr(kl_out), _stream()), 'ppo_loss_finalize')


def mask_inv_counts(mask, H, N, envs_per_mb, inv_count):
    check(lib.b200rl_mask_inv_counts_f32(ptr(mask), H, N, envs_per_mb, ptr(inv_count), _stream()), 'mask_inv_counts')


class PackTable(ctypes.Structure):
    _fields_ = [('n_seg', ctypes.c_int), ('flat_off', ctypes.c_int * 4), ('rows', ctypes.c_int * 4), ('cols', ctypes.c_int * 4),
                ('cs_bytes', ctypes.c_uint32 * 4), ('dst_off', ctypes.c_uint32 * 4)]


class ObsMerge(ctypes.Structure):
    _fields_ = [('mbmom', ctypes.c_void_p), ('shift', ctypes.c_void_p), ('D', ctypes.c_int), ('n_rows', ctypes.c_int),
                ('mean', ctypes.c_void_p), ('var', ctypes.c_void_p), ('count', ctypes.c_void_p), ('mean_f32', ctypes.c_void_p),
                ('std_f32', ctypes.c_void_p), ('eps', ctypes.c_float)]


def make_obs_merge(mbmom_i, shift, D, n_rows, mean, var, count, mean_f32, std_f32, eps=1e-5):
    return ObsMerge(ptr(mbmom_i), ptr(shift), D, n_rows, ptr(mean), ptr(var), ptr(count), ptr(mean_f32), ptr(std_f32), eps)


def lr_schedule_apply(state_d, kl_dev, kl_scale, base_lr, cfg):
    check(lib.b200rl_lr_schedule_apply(ptr(state_d), ptr(kl_dev), float(kl_scale), float(base_lr), ctypes.addressof(cfg), _stream()),
          'lr_schedule_apply')


def adam_step(params, grads, exp_avg, exp_avg_sq, state_d, kl_dev, cfg, stats_out, counter, n=None, wpack=None, pack_table=None,
              merge_next=None):
    check(lib.b200rl_adam_step_f32(ptr(params), ptr(grads), ptr(exp_avg), ptr(exp_avg_sq),
                                   params.numel() if n is None else n, ptr(state_d), ptr(kl_dev), ctypes.addressof(cfg),
                                   ptr(stats_out), ptr(counter), ptr(wpack),
                                   None if pack_table is None else ctypes.addressof(pack_table),
                                   None if merge_next is None else ctypes.addressof(merge_next), _stream()), 'adam_step')


def reduce_finalize(part, out, n, n_splits, split_stride, partials, n_partials, A, entropy_coef_dev, stats, d_logstd, kl_out=None):
    check(lib.b200rl_reduce_finalize(ptr(part), ptr(out), n, n_splits, split_stride, ptr(partials), n_partials, A,
                                     ptr(entropy_coef_dev), ptr(stats), ptr(d_logstd), ptr(kl_out), _stream()), 'reduce_finalize')


def reduce_adam(part, n_splits, split_stride, loss_partials, n_loss_partials, A, entropy_coef_dev, stats, kl_out, grads, params,
                exp_avg, exp_avg_sq, n, state_d, cfg, counter, nrm_part, grid_bar, wpack=None, pack_table=None, merge_next=None):
    """single-GPU fused minibatch tail: split reduce + loss finalise + clip + Adam in one launch"""
    check(lib.b200rl_reduce_adam_f32(ptr(part), n_splits, split_stride, ptr(loss_partials), n_loss_partials, A, ptr(entropy_coef_dev),
                                     ptr(stats), ptr(kl_out), ptr(grads), ptr(params), ptr(exp_avg), ptr(exp_avg_sq), n, ptr(state_d),
                                     ctypes.addressof(cfg), ptr(counter), ptr(nrm_part), nrm_part.numel(), ptr(grid_bar), ptr(wpack),
                                     None if pack_table is None else ctypes.addressof(pack_table),
                                     None if merge_next is None else ctypes.addressof(merge_next), _stream()), 'reduce_adam')


def tc_pack_table(D, units, A, offs):
    t = PackTable()
    check(lib.b200rl_tc_pack_table(D, units[0], units[1], units[2], A, offs['W0'], offs['W1'], offs['W2'], offs['W_head'],
                                   ctypes.addressof(t)), 'tc_pack_table')
    return t


def policy_head_sample(a_last, W_head, b_head, logstd, vms_mean, vms_var, normalize_value, noise, seed, rng_epoch,
                       step_index, actions, mus, sigmas, neglogp, values, env_actions, clip_actions, act_low, act_high,
                       dones_cur, dones_out, prev_dones, valid_out, N, A, values_only=False):
    Hl = W_head.shape[1]
    check(lib.b200rl_policy_head_sample_f32(ptr(a_last), Hl, ptr(W_head), ptr(b_head), ptr(logstd), ptr(vms_mean),
                                            ptr(vms_var), int(normalize_value), ptr(noise), seed, ptr(rng_epoch),
                                            step_index, ptr(actions), ptr(mus), ptr(sigmas), ptr(neglogp), ptr(values),
                                            ptr(env_actions), int(clip_actions), ptr(act_low), ptr(act_high),
                                            ptr(dones_cur), ptr(dones_out), ptr(prev_dones), ptr(valid_out), N, A,
                                            int(values_only), _stream()), 'policy_head_sample')


def post_step(rewards, dones, time_outs, values_t, valid_t, rewards_out_t, dones_cur, prev_dones, ep_state, meter,
              games_to_track, scratch, counter, N, cfg):
    d_u8 = 1 if dones.dtype in (torch.uint8, torch.bool) else 0
    if not d_u8 and dones.dtype != torch.float32:
        dones = dones.float()
    kind = 0
    if time_outs is not None:
        if time_outs.dtype in (torch.uint8, torch.bool):
            kind = 1
        else:
            kind = 2
            if time_outs.dtype != torch.float32:
                time_outs = time_outs.float()
    check(lib.b200rl_post_step_f32(ptr(rewards), ptr(dones), d_u8, ptr(time_outs), kind, ptr(values_t), ptr(valid_t),
                                   ptr(rewards_out_t), ptr(dones_cur), ptr(prev_dones), ptr(ep_state), ptr(meter),
                                   games_to_track, ptr(scratch), scratch.numel() // 4, ptr(counter), N,
                                   ctypes.addressof(cfg), _stream()), 'post_step')


def synth_env_step(actions, obs, rewards, dones, time_outs, ep_t, N, D, A, max_len, p_done, seed, rng_epoch, step_index):
    check(lib.b200rl_synth_env_step(ptr(actions), ptr(obs), ptr(rewards), ptr(dones), ptr(time_outs), ptr(ep_t), N, D, A,
                                    max_len, p_done, seed, ptr(rng_epoch), step_index, _stream()), 'synth_env_step')


def bump_u64(t):
    check(lib.b200rl_bump_u64(ptr(t), _stream()), 'bump_u64')


def fill_u32(t, v=0):
    check(lib.b200rl_fill_u32(ptr(t), t.numel() * t.element_size() // 4, v, _stream()), 'fill_u32')


def tc_gemm_test(A, B, N, K, a_mn=False, b_mn=False):
    D = torch.empty(128, N, dtype=torch.float32, device=A.device)
    check(lib.b200rl_tc_gemm_test(ptr(A), ptr(B), ptr(D), N, K, int(a_mn), int(b_mn), _stream()), 'tc_gemm_test')
    return D


# ------------------------------------------------------------------------------------------ bf16 tcgen05 path
def tc_kind(D, units, A):
    """0 = no tcgen05 kernels for this geometry, 1 = resident-weights kernels (obs <= 64), 2 = wide observations (64 < obs <= 256)"""
    return int(lib.b200rl_tc_supported(D, units[0], units[1], units[2], A)) if len(units) == 3 else 0


def tc_supported(D, units, A, allow_wide=False):
    k = tc_kind(D, units, A)
    return k == 1 or (allow_wide and k == 2)


def tc_pack_bytes(D, units, A):
    return int(lib.b200rl_tc_pack_bytes(D, units[0], units[1], units[2], A))


def tc_tile_bytes(D, units, A):
    out = (ctypes.c_int64 * 4)()
    check(lib.b200rl_tc_tile_bytes(D, units[0], units[1], units[2], A, ctypes.addressof(out)), 'tc_tile_bytes')
    return [int(x) for x in out]


def set_pdl(enable):
    """programmatic dependent launch of the chain kernels (process-wide); returns the previous setting"""
    return bool(lib.b200rl_set_pdl(int(bool(enable))))


def tc_xtile_bytes(D, units, A):
    n = int(lib.b200rl_tc_xtile_bytes(D, units[0], units[1], units[2], A))
    if n < 0:
        raise B200RLError('tc_xtile_bytes: unsupported geometry')
    return n


def tc_pack_weights(W1, W2, W3, W_head, D, units, A, wpack):
    check(lib.b200rl_tc_pack_weights(ptr(W1), ptr(W2), ptr(W3), ptr(W_head), D, units[0], units[1], units[2], A, ptr(wpack),
                                     _stream()), 'tc_pack_weights')


def tc_mlp_fwd_train(obs, rows_per_chunk, chunk_stride, D, nm, ns, wpack, b, b_head, logstd, units, M, A, actions, old_mu,
                     old_sigma, old_values_n, returns_n, old_neglogp, advs_n, mask, cfg, inv_count, act, dhead, partials, xtile=None,
                     activation=1):
    nb = ctypes.c_int(0)
    check(lib.b200rl_tc_mlp_fwd_train(ptr(obs), rows_per_chunk, chunk_stride, D, ptr(nm), ptr(ns), ptr(wpack), ptr(b[0]), ptr(b[1]),
                                      ptr(b[2]), ptr(b_head), ptr(logstd), units[0], units[1], units[2], int(activation), M, A, ptr(actions),
                                      ptr(old_mu), ptr(old_sigma), ptr(old_values_n), ptr(returns_n), ptr(old_neglogp), ptr(advs_n),
                                      ptr(mask), ctypes.addressof(cfg), ptr(inv_count), ptr(act[0]), ptr(act[1]), ptr(act[2]),
                                      ptr(dhead), ptr(xtile), ptr(partials), partials.shape[0], ctypes.addressof(nb), _stream()),
          'tc_mlp_fwd_train')
    return nb.value


def tc_mlp_fwd_rollout(obs, D, nm, ns, wpack, b, b_head, logstd, units, N, A, vms_mean, vms_var, normalize_value, noise, seed,
                       rng_epoch, step_index, actions, mus, sigmas, neglogp, values, env_actions, clip_actions, act_low, act_high,
                       dones_cur, dones_out, prev_dones, valid_out, values_only=False, l1_scratch=None, activation=1):
    check(lib.b200rl_tc_mlp_fwd_rollout(ptr(obs), D, ptr(nm), ptr(ns), ptr(wpack), ptr(b[0]), ptr(b[1]), ptr(b[2]), ptr(b_head),
                                        ptr(logstd), units[0], units[1], units[2], int(activation), N, A, ptr(vms_mean), ptr(vms_var),
                                        int(normalize_value), ptr(noise), seed, ptr(rng_epoch), step_index, ptr(actions), ptr(mus),
                                        ptr(sigmas), ptr(neglogp), ptr(values), ptr(env_actions), int(clip_actions), ptr(act_low),
                                        ptr(act_high), ptr(dones_cur), ptr(dones_out), ptr(prev_dones), ptr(valid_out),
                                        int(values_only), ptr(l1_scratch), _stream()), 'tc_mlp_fwd_rollout')


def tc_mlp_bwd(obs, rows_per_chunk, chunk_stride, D, nm, ns, wpack, units, M, A, act, dhead, delta2, delta1, part, P, offs,
               xtile=None, activation=1, pipelined_wgrad=False):
    """offs: dict with W0,b0,W1,b1,W2,b2,W_head,b_head flat offsets (model.layout)."""
    nb = ctypes.c_int(0)
    check(lib.b200rl_tc_mlp_bwd(ptr(obs), rows_per_chunk, chunk_stride, D, ptr(nm), ptr(ns), ptr(wpack), units[0], units[1], units[2],
                                int(activation), M, A, ptr(act[0]), ptr(act[1]), ptr(act[2]), ptr(dhead), ptr(xtile), int(pipelined_wgrad), ptr(delta2), ptr(delta1), ptr(part),
                                part.shape[0], P, offs['W0'], offs['b0'], offs['W1'], offs['b1'], offs['W2'], offs['b2'],
                                offs['W_head'], offs['b_head'], ctypes.addressof(nb), _stream()), 'tc_mlp_bwd')
    return nb.value


# ------------------------------------------------------------------------------------------ multi-GPU peer memory
def ipc_alloc(nbytes):
    p = ctypes.c_void_p()
    h = (ctypes.c_ubyte * 64)()
    check(lib.b200rl_ipc_alloc(nbytes, ctypes.addressof(p), ctypes.addressof(h)), 'ipc_alloc')
    return p.value, bytes(h)


def ipc_open(handle):
    p = ctypes.c_void_p()
    h = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
    check(lib.b200rl_ipc_open(ctypes.addressof(h), ctypes.addressof(p)), 'ipc_open')
    return p.value


class _RawCuda:
    def __init__(self, ptr_, shape, typestr):
        self.__cuda_array_interface__ = {'shape': tuple(shape), 'typestr': typestr, 'data': (int(ptr_), False), 'version': 2}


def tensor_from_ptr(ptr_, n, dtype, device):
    typestr = {torch.float32: '<f4', torch.int64: '<i8', torch.uint8: '|u1'}[dtype]
    return torch.as_tensor(_RawCuda(ptr_, (n,), typestr), device=device)


class PeerTable:
    """host-side pointer tables handed to b200rl_allreduce_adam_f32"""

    def __init__(self, grads_ptrs, flags_ptrs, cta_flags_ptrs=None):
        self.world = len(flags_ptrs)
        self.grads = [(ctypes.c_void_p * 8)(*(list(g) + [None] * (8 - len(g)))) for g in grads_ptrs]   # one table per parity
        self.flags = (ctypes.c_void_p * 8)(*(list(flags_ptrs) + [None] * (8 - len(flags_ptrs))))
        cf = list(cta_flags_ptrs) if cta_flags_ptrs is not None else []
        self.cta_flags = (ctypes.c_void_p * 8)(*(cf + [None] * (8 - len(cf))))      # per-CTA flag arrays (reduce_allreduce_adam)


def allreduce_adam(table, parity, rank, my_flags_ptr, seq, red, nrm_part, grid_bar, params, exp_avg, exp_avg_sq, n, state_d, cfg,
                   stats_out, counter, wpack=None, pack_table=None, merge_next=None):
    check(lib.b200rl_allreduce_adam_f32(ctypes.addressof(table.grads[parity]), ctypes.addressof(table.flags), table.world, rank,
                                        my_flags_ptr, ptr(seq), ptr(red), ptr(nrm_part), nrm_part.numel(), ptr(grid_bar), ptr(params),
                                        ptr(exp_avg), ptr(exp_avg_sq), n, ptr(state_d), ctypes.addressof(cfg), ptr(stats_out),
                                        ptr(counter), ptr(wpack), None if pack_table is None else ctypes.addressof(pack_table),
                                        None if merge_next is None else ctypes.addressof(merge_next), _stream()), 'allreduce_adam')


PEER_FLAG_STRIDE = 160      # B200RL_PEER_FLAG_STRIDE


def reduce_allreduce_adam(part, n_splits, split_stride, loss_partials, n_loss_partials, A, entropy_coef_dev, stats, table, parity, rank,
                          my_cta_flags_ptr, seq, red, params, exp_avg, exp_avg_sq, n, state_d, cfg, counter, nrm_part, grid_bar,
                          wpack=None, pack_table=None, merge_next=None):
    """multi-GPU fused minibatch tail: split reduce + loss finalise + peer-memory all-reduce + clip + Adam in one launch"""
    check(lib.b200rl_reduce_allreduce_adam_f32(ptr(part), n_splits, split_stride, ptr(loss_partials), n_loss_partials, A,
                                               ptr(entropy_coef_dev), ptr(stats), ctypes.addressof(table.grads[parity]),
                                               ctypes.addressof(table.cta_flags), table.world, rank, my_cta_flags_ptr, ptr(seq), ptr(red),
                                               ptr(params), ptr(exp_avg), ptr(exp_avg_sq), n, ptr(state_d), ctypes.addressof(cfg),
                                               ptr(counter), ptr(nrm_part), nrm_part.numel(), ptr(grid_bar), ptr(wpack),
                                               None if pack_table is None else ctypes.addressof(pack_table),
                                               None if merge_next is None else ctypes.addressof(merge_next), _stream()),
          'reduce_allreduce_adam')


# ------------------------------------------------------------------------------------------ LSTM cell (fp32)
def lstm_cell_fwd(gates, cin, c_out, h_out, S, Hd, h_scatter=None, scatter_rpc=0, scatter_stride=0, hin_next=None, cin_next=None,
                  done_next=None, done_rpc=0, done_stride=0):
    check(lib.b200rl_lstm_cell_fwd_f32(ptr(gates), ptr(cin), ptr(c_out), ptr(h_out), ptr(h_scatter), scatter_rpc, scatter_stride,
                                       ptr(hin_next), ptr(cin_next), ptr(done_next), done_rpc, done_stride, S, Hd, _stream()),
          'lstm_cell_fwd')


def lstm_cell_bwd(gates_act, c_t, cin, dgates, dcin, S, Hd, dH=None, scatter_rpc=0, scatter_stride=0, dhin_next=None, dcin_next=None,
                  done_next=None, done_rpc=0, done_stride=0):
    check(lib.b200rl_lstm_cell_bwd_f32(ptr(gates_act), ptr(c_t), ptr(cin), ptr(dH), scatter_rpc, scatter_stride, ptr(dhin_next),
                                       ptr(dcin_next), ptr(done_next), done_rpc, done_stride, ptr(dgates), ptr(dcin), S, Hd, _stream()),
          'lstm_cell_bwd')


def rnn_train_dones(dones_u8, valid, out_u8):
    H, N = dones_u8.shape
    check(lib.b200rl_rnn_train_dones_u8(ptr(dones_u8), ptr(valid), ptr(out_u8), H, N, _stream()), 'rnn_train_dones')


def rnn_mask_rows(inp, in_rpc, in_stride, out, S, Hd, done=None, done_rpc=0, done_stride=0):
    check(lib.b200rl_rnn_mask_rows_f32(ptr(inp), in_rpc, in_stride, ptr(out), ptr(done), done_rpc, done_stride, S, Hd, _stream()),
          'rnn_mask_rows')


# ------------------------------------------------------------------------------------------ categorical head (discrete PPO; csrc/discrete.cu)
class CatLossCfg(ctypes.Structure):
    _fields_ = [('e_clip', ctypes.c_float), ('critic_coef', ctypes.c_float), ('entropy_coef', ctypes.c_float),
                ('clip_value', ctypes.c_int), ('use_smooth_clamp', ctypes.c_int), ('ppo', ctypes.c_int)]


def _head_table(head_sizes):
    if not head_sizes:
        return 0, None
    arr = (ctypes.c_int * len(head_sizes))(*[int(k) for k in head_sizes])
    return len(head_sizes), arr


def categorical_sample(logits, ld, K, value_raw, value_ld, action_masks, u_tape, seed, rng_epoch, step_index, vms_mean, vms_var,
                       normalize_value, actions, neglogp, values, dones_cur, dones_out, prev_dones, valid_out, N, values_only=False,
                       head_sizes=None):
    """head_sizes: sizes of the heads of a multi-discrete (Tuple) space (sum = K; actions [N, n_heads], u_tape [n_heads, N]); None = one head"""
    nh, tab = _head_table(head_sizes)
    check(lib.b200rl_categorical_sample_f32(ptr(logits), ld, K, nh, None if tab is None else ctypes.addressof(tab), ptr(value_raw), value_ld,
                                            ptr(action_masks), ptr(u_tape), seed, ptr(rng_epoch), step_index, ptr(vms_mean), ptr(vms_var),
                                            int(normalize_value), ptr(actions), ptr(neglogp), ptr(values), ptr(dones_cur), ptr(dones_out),
                                            ptr(prev_dones), ptr(valid_out), N, int(values_only), _stream()), 'categorical_sample')


def categorical_loss(logits, ld, K, values, value_ld, actions, action_masks, old_values_n, returns_n, old_neglogp, advs_n, mask,
                     rows_per_chunk, chunk_stride, M, cfg, inv_count, d_logits, d_ld, d_value, dv_ld, partials, head_sizes=None):
    nb = ctypes.c_int(0)
    nh, tab = _head_table(head_sizes)
    check(lib.b200rl_categorical_loss_f32(ptr(logits), ld, K, nh, None if tab is None else ctypes.addressof(tab), ptr(values), value_ld,
                                          ptr(actions), ptr(action_masks), ptr(old_values_n), ptr(returns_n), ptr(old_neglogp), ptr(advs_n),
                                          ptr(mask), rows_per_chunk, chunk_stride, M, ctypes.addressof(cfg), ptr(inv_count), ptr(d_logits),
                                          d_ld, ptr(d_value), dv_ld, ptr(partials), partials.shape[0], ctypes.addressof(nb), _stream()),
          'categorical_loss')
    return nb.value


def value_loss(values, value_ld, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count, d_value, dv_ld,
               partials):
    """central-value critic loss + gradient (csrc/critic.cu)"""
    nb = ctypes.c_int(0)
    check(lib.b200rl_value_loss_f32(ptr(values), value_ld, ptr(old_values_n), ptr(returns_n), ptr(mask), rows_per_chunk, chunk_stride, M,
                                    float(e_clip), int(clip_value), ptr(inv_count), ptr(d_value), dv_ld, ptr(partials), partials.shape[0],
                                    ctypes.addressof(nb), _stream()), 'value_loss')
    return nb.value


VALUE_HEAD_MAX_HL = 4096        # B200RL_VALUE_HEAD_MAX_HL


def value_head_loss(a_last, W_v, b_v, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count, act_last,
                    d_alast, dW_part, db_part, split_stride, n_splits, partials, value_out=None):
    """fused value head of the tensor-core critic (csrc/critic.cu): value GEMV + value_loss + d(a_last) + head gradient split rows"""
    nb = ctypes.c_int(0)
    check(lib.b200rl_value_head_loss_f32(ptr(a_last), W_v.numel(), ptr(W_v), ptr(b_v), ptr(old_values_n), ptr(returns_n), ptr(mask),
                                         rows_per_chunk, chunk_stride, M, float(e_clip), int(clip_value), ptr(inv_count), act_last,
                                         ptr(d_alast), ptr(value_out), ptr(dW_part), ptr(db_part), split_stride, n_splits, ptr(partials),
                                         partials.shape[0], ctypes.addressof(nb), _stream()), 'value_head_loss')
    return nb.value


def value_head_fwd(a_last, W_v, b_v, vms_mean, vms_var, normalize_value, values, N):
    """rollout value of the tensor-core critic: values[N] = denorm(W_v . a_last + b_v) in one launch"""
    check(lib.b200rl_value_head_fwd_f32(ptr(a_last), W_v.numel(), ptr(W_v), ptr(b_v), ptr(vms_mean), ptr(vms_var), int(normalize_value),
                                        ptr(values), N, _stream()), 'value_head_fwd')
