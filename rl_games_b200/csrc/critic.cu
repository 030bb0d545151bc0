// Value-only loss head of the central value network (asymmetric critic) -- SURVEY.md 8f rank 1 (algos_torch/central_value.py:276-301
// calc_loss / calc_gradients: loss = masked mean of common_losses.critic_loss).
//
// The per-row arithmetic is __host__ __device__ and is also exercised on the CPU (tests/test_critic_rows_cpu.py); GPU parity:
// tests/test_cv_gpu.py.
//
// The tensor-core critic (central_value_config mixed_precision: True) replaces the four launches of its 1-wide value head (linear_fwd,
// value_loss, linear_bwd_weight, linear_bwd_data) with value_head_loss_kernel, and its rollout head (linear_fwd + normalize) with
// value_head_fwd_kernel (GPU checks: tests/test_cv_tensor_cores_gpu.py).
#include <cooperative_groups.h>

#include "common.cuh"

namespace {

// critic_loss of one row (common_losses.py:7-38) and d(loss)/d(value); returns the loss
__host__ __device__ inline float value_loss_row(float val, float old_v, float ret, float e_clip, int clip_value, float& dc) {
    if (clip_value) {
        const float delta = val - old_v;
        const float vpc = old_v + fminf(fmaxf(delta, -e_clip), e_clip);
        const float e1 = val - ret, e2 = vpc - ret;
        const float l1 = e1 * e1, l2 = e2 * e2;
        const float g1 = 2.0f * e1, g2 = (delta >= -e_clip && delta <= e_clip) ? 2.0f * e2 : 0.0f;
        dc = (l1 > l2) ? g1 : ((l1 < l2) ? g2 : 0.5f * (g1 + g2));
        return fmaxf(l1, l2);
    }
    const float e1 = ret - val;
    dc = -2.0f * e1;
    return e1 * e1;
}

struct ValueLossArgs {
    const float* values; int value_ld; const float* old_values_n; const float* returns_n; const float* mask; int rows_per_chunk;
    int64_t chunk_stride; int M; float e_clip; int clip_value; const float* inv_count_dev; float* d_value; int dv_ld;
};

// everything one kernel thread does except the block reduction (__host__ __device__: the arena addressing runs on the CPU too,
// b200rl_hosttest_value_loss_arena).  acc: sum w*c_loss, sum mask, sum w
__host__ __device__ inline void value_loss_thread(const ValueLossArgs& a, int m, double (&acc)[3]) {
    const int c = m / a.rows_per_chunk;
    const int64_t ar = (int64_t)c * a.chunk_stride + (m - c * a.rows_per_chunk);
    const float mk = a.mask ? a.mask[ar] : 1.0f;
    const float w = mk * (a.inv_count_dev ? a.inv_count_dev[0] : (1.0f / (float)a.M));
    float dc;
    const float l = value_loss_row(a.values[(int64_t)m * a.value_ld], a.old_values_n[ar], a.returns_n[ar], a.e_clip, a.clip_value, dc);
    a.d_value[(int64_t)m * a.dv_ld] = w * dc;
    acc[0] = (double)w * l; acc[1] = mk; acc[2] = w;
}

// partial row (8 doubles per block): sum w*c_loss, sum mask, sum w, 0...
__global__ void __launch_bounds__(256) value_loss_kernel(const ValueLossArgs a, double* __restrict__ partials) {
    __shared__ double sm[32 * 3];
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    double acc[3] = {0, 0, 0};
    if (m < a.M) value_loss_thread(a, m, acc);
    block_sum_d<3>(acc, sm);
    if (threadIdx.x == 0) {
        double* p = partials + (int64_t)blockIdx.x * 8;
        p[0] = acc[0]; p[1] = acc[1]; p[2] = acc[2];
#pragma unroll
        for (int i = 3; i < 8; ++i) p[i] = 0.0;
    }
}

// value_loss_thread for a value the caller already holds (the fused head computes it itself): same chunk mapping, weight and loss
// arithmetic; returns d(loss)/d(value) of row m
__host__ __device__ inline float value_head_thread(const ValueLossArgs& a, int m, float val, double (&acc)[3]) {
    const int c = m / a.rows_per_chunk;
    const int64_t ar = (int64_t)c * a.chunk_stride + (m - c * a.rows_per_chunk);
    const float mk = a.mask ? a.mask[ar] : 1.0f;
    const float w = mk * (a.inv_count_dev ? a.inv_count_dev[0] : (1.0f / (float)a.M));
    float dc;
    const float l = value_loss_row(val, a.old_values_n[ar], a.returns_n[ar], a.e_clip, a.clip_value, dc);
    acc[0] = (double)w * l; acc[1] = mk; acc[2] = w;
    return w * dc;
}

// ---- fused value head of the tensor-core critic: v = W_v . a_last + b_v (fp32), loss, d(a_last) and the head's weight gradient ----
// One cluster of C CTAs per gradient split s owns the split's rows [s*rps, (s+1)*rps) (rps a multiple of 256); CTA c of the cluster
// takes the split's 256-row tiles c, c+C, ...  A tile is one loss partial row, exactly as value_loss_kernel's 256-thread blocks.
// The head gradient is summed per warp (lane-owned columns in shared memory), then over the 8 warps, then over the cluster's CTAs
// through distributed shared memory, each in a fixed order: deterministic, no atomics.
constexpr int VH_THREADS = 256, VH_WARPS = VH_THREADS / 32, VH_MAX_CLUSTER = 8;

// the dot product of one row, lanes striding over k; every lane returns the full sum (identical in the rollout and training kernels)
__device__ __forceinline__ float vh_row_dot(const float* __restrict__ a, const float* w, int Hl, int lane) {
    float d = 0.f;
    for (int k = lane; k < Hl; k += 32) d = fmaf(a[k], w[k], d);
    return warp_sum(d);
}

struct ValueHeadArgs {
    ValueLossArgs l;                         // loss operands (values / d_value unused)
    const float* a_last; int Hl; const float* W_v; const float* b_v; int act_last;
    float* d_alast; float* value_out; float* dW_part; float* db_part; int64_t split_stride; int rows_per_split;
};

__global__ void __launch_bounds__(VH_THREADS) value_head_loss_kernel(const ValueHeadArgs p, double* __restrict__ partials) {
    namespace cg = cooperative_groups;
    extern __shared__ float vh_smem[];
    __shared__ float sv[VH_THREADS], sdv[VH_THREADS], sdb[VH_WARPS];
    __shared__ double sm[32 * 3];
    const int Hl = p.Hl, M = p.l.M, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* sW = vh_smem;                       // [Hl] the head's weights
    float* sdw = vh_smem + Hl;                 // [VH_WARPS][Hl] per-warp weight-gradient sums; row 0 ends as the CTA's sum
    const cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks(), c = (int)cluster.block_rank(), s = blockIdx.y;
    for (int k = tid; k < Hl; k += VH_THREADS) sW[k] = p.W_v[k];
    for (int k = tid; k < VH_WARPS * Hl; k += VH_THREADS) sdw[k] = 0.f;
    if (tid < VH_WARPS) sdb[tid] = 0.f;
    const float bv = p.b_v[0];
    const int s0 = min((int64_t)s * p.rows_per_split, (int64_t)M), s1 = min((int64_t)s0 + p.rows_per_split, (int64_t)M);
    __syncthreads();
    for (int m0 = s0 + c * VH_THREADS; m0 < s1; m0 += C * VH_THREADS) {
        const int nr = min(VH_THREADS, s1 - m0);
        // 1) values: warp w computes rows 32w .. 32w+31, four at a time
        for (int r = warp * 32; r < warp * 32 + 32; r += 4) {
            float d[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) d[j] = 0.f;
            for (int k = lane; k < Hl; k += 32) {
                const float wk = sW[k];
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (r + j < nr) d[j] = fmaf(p.a_last[(int64_t)(m0 + r + j) * Hl + k], wk, d[j]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                d[j] = warp_sum(d[j]);
                if (lane == 0) sv[r + j] = d[j] + bv;
            }
        }
        __syncthreads();
        // 2) loss and d(loss)/d(value), one row per thread (value_loss_kernel's arithmetic and partial row)
        double acc[3] = {0, 0, 0};
        float dv = 0.f;
        if (tid < nr) {
            dv = value_head_thread(p.l, m0 + tid, sv[tid], acc);
            if (p.value_out) p.value_out[m0 + tid] = sv[tid];
        }
        sdv[tid] = dv;
        block_sum_d<3>(acc, sm);                 // its barriers also publish sdv
        if (tid == 0) {
            double* q = partials + (int64_t)(m0 / VH_THREADS) * 8;
            q[0] = acc[0]; q[1] = acc[1]; q[2] = acc[2];
#pragma unroll
            for (int i = 3; i < 8; ++i) q[i] = 0.0;
        }
        // 3) d(a_last) = d_v * W_v * act'(a_last) and the head gradient, warp w on its own rows
        float* dw = sdw + warp * Hl;
        for (int r = warp * 32; r < min(warp * 32 + 32, nr); ++r) {
            const float g = sdv[r];
            const int64_t row = (int64_t)(m0 + r) * Hl;
            for (int k = lane; k < Hl; k += 32) {
                const float av = p.a_last[row + k];
                p.d_alast[row + k] = (g * sW[k]) * act_bwd_from_out(av, p.act_last);
                dw[k] = fmaf(g, av, dw[k]);
            }
            if (lane == 0) sdb[warp] += g;
        }
        __syncthreads();                         // sv / sdv are rewritten by the next tile
    }
    // 4) CTA sum over the warps (fixed order) into sdw row 0, then the cluster's rank 0 sums the CTAs (fixed order) into split s
    for (int k = tid; k < Hl; k += VH_THREADS) {
        float t = sdw[k];
        for (int w = 1; w < VH_WARPS; ++w) t += sdw[w * Hl + k];
        sdw[k] = t;
    }
    if (tid == 0) {
        float t = sdb[0];
        for (int w = 1; w < VH_WARPS; ++w) t += sdb[w];
        sdb[0] = t;
    }
    cluster.sync();
    if (c == 0) {
        float* dW = p.dW_part + (int64_t)s * p.split_stride;
        for (int k = tid; k < Hl; k += VH_THREADS) {
            float t = sdw[k];
            for (int q = 1; q < C; ++q) t += cluster.map_shared_rank(sdw, q)[k];
            dW[k] = t;
        }
        if (tid == 0) {
            float t = sdb[0];
            for (int q = 1; q < C; ++q) t += cluster.map_shared_rank(sdb, q)[0];
            p.db_part[(int64_t)s * p.split_stride] = t;
        }
    }
    cluster.sync();                              // the other CTAs' shared memory stays alive until rank 0 has read it
}

// rollout: values[n] = denorm(W_v . a_last[n] + b_v), one warp per row; the de-normalisation is normalize_kernel's (denorm = 1)
__global__ void __launch_bounds__(256) value_head_fwd_kernel(const float* __restrict__ a_last, int Hl, const float* __restrict__ W_v,
                                                             const float* __restrict__ b_v, const double* __restrict__ vms_mean,
                                                             const double* __restrict__ vms_var, int normalize_value,
                                                             float* __restrict__ values, int N) {
    const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    float v = vh_row_dot(a_last + (int64_t)n * Hl, W_v, Hl, lane) + b_v[0];
    if (lane == 0) {
        if (normalize_value) {
            const float m = (float)vms_mean[0];
            const float sd = __fsqrt_rn(__fadd_rn((float)vms_var[0], 1e-5f));
            v = __fadd_rn(__fmul_rn(sd, fminf(fmaxf(v, -5.0f), 5.0f)), m);
        }
        values[n] = v;
    }
}

}  // namespace

B200RL_EXPORT int b200rl_value_loss_f32(const float* values, int value_ld, const float* old_values_n, const float* returns_n,
                                        const float* mask, int rows_per_chunk, int64_t chunk_stride, int M, float e_clip, int clip_value,
                                        const float* inv_count_dev, float* d_value, int dv_ld, double* partials, int max_partials,
                                        int* n_blocks_out_host, void* stream) {
    if (!values || !old_values_n || !returns_n || !d_value || !partials || M <= 0 || value_ld <= 0 || dv_ld <= 0 || rows_per_chunk <= 0)
        return B200RL_EINVAL;
    const int blocks = (M + 255) / 256;
    if (n_blocks_out_host) *n_blocks_out_host = blocks;
    if (blocks > max_partials) return B200RL_EINVAL;
    const ValueLossArgs a{values, value_ld, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count_dev,
                          d_value, dv_ld};
    value_loss_kernel<<<blocks, 256, 0, as_stream(stream)>>>(a, partials);
    B200RL_LAUNCH_CHECK();
    return B200RL_OK;
}

B200RL_EXPORT int b200rl_value_head_loss_f32(const float* a_last, int Hl, const float* W_v, const float* b_v, const float* old_values_n,
                                             const float* returns_n, const float* mask, int rows_per_chunk, int64_t chunk_stride, int M,
                                             float e_clip, int clip_value, const float* inv_count_dev, int act_last, float* d_alast,
                                             float* value_out, float* dW_part, float* db_part, int64_t split_stride, int n_splits,
                                             double* partials, int max_partials, int* n_blocks_out_host, void* stream) {
    if (!a_last || !W_v || !b_v || !old_values_n || !returns_n || !d_alast || !dW_part || !db_part || !partials || Hl <= 0 || M <= 0 ||
        rows_per_chunk <= 0 || n_splits <= 0 || n_splits > 65535 || split_stride < Hl)
        return B200RL_EINVAL;
    if (Hl > B200RL_VALUE_HEAD_MAX_HL) return B200RL_EUNSUPPORTED;
    const int blocks = (M + VH_THREADS - 1) / VH_THREADS;
    if (n_blocks_out_host) *n_blocks_out_host = blocks;
    if (blocks > max_partials) return B200RL_EINVAL;
    const int rps = ((M + n_splits - 1) / n_splits + VH_THREADS - 1) / VH_THREADS * VH_THREADS;
    const int C = min(VH_MAX_CLUSTER, rps / VH_THREADS);
    const size_t smem = (size_t)(1 + VH_WARPS) * Hl * sizeof(float);
    static size_t smem_set = 0;
    if (smem > 48 * 1024 && smem > smem_set) {
        const cudaError_t e = cudaFuncSetAttribute(value_head_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        smem_set = smem;
    }
    const ValueHeadArgs p{{nullptr, 1, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count_dev,
                           nullptr, 1},
                          a_last, Hl, W_v, b_v, act_last, d_alast, value_out, dW_part, db_part, split_stride, rps};
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(C, n_splits, 1); cfg.blockDim = dim3(VH_THREADS, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = as_stream(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, value_head_loss_kernel, p, partials);
    if (e != cudaSuccess) return (int)e;
    B200RL_LAUNCH_CHECK();
    return B200RL_OK;
}

B200RL_EXPORT int b200rl_value_head_fwd_f32(const float* a_last, int Hl, const float* W_v, const float* b_v, const double* vms_mean,
                                            const double* vms_var, int normalize_value, float* values, int N, void* stream) {
    if (!a_last || !W_v || !b_v || !values || Hl <= 0 || N <= 0 || (normalize_value && (!vms_mean || !vms_var))) return B200RL_EINVAL;
    value_head_fwd_kernel<<<(N + 7) / 8, 256, 0, as_stream(stream)>>>(a_last, Hl, W_v, b_v, vms_mean, vms_var, normalize_value, values, N);
    B200RL_LAUNCH_CHECK();
    return B200RL_OK;
}

#ifdef B200RL_TEST_HOOKS   // test-only host entry points: compiled into tests/libb200rl_testhooks.so (csrc/build.py), not into the product library
// host test entry point (CPU, host arrays): the same row function; not declared in include/b200rl.h, never called by the product
B200RL_EXPORT int b200rl_hosttest_value_loss_rows(const float* values, const float* old_values_n, const float* returns_n, const float* w,
                                                 int M, float e_clip, int clip_value, float* d_value, double* loss_sum) {
    double s = 0.0;
    for (int m = 0; m < M; ++m) {
        float dc;
        const float l = value_loss_row(values[m], old_values_n[m], returns_n[m], e_clip, clip_value, dc);
        d_value[m] = w[m] * dc;
        s += (double)w[m] * l;
    }
    *loss_sum = s;
    return B200RL_OK;
}

// the kernel's per-thread body over HOST arrays laid out like the device arena (arguments of the C-ABI entry point, no stream)
B200RL_EXPORT int b200rl_hosttest_value_loss_arena(const float* values, int value_ld, const float* old_values_n, const float* returns_n,
                                                  const float* mask, int rows_per_chunk, int64_t chunk_stride, int M, float e_clip, int clip_value,
                                                  const float* inv_count, float* d_value, int dv_ld, double* partial8) {
    const ValueLossArgs a{values, value_ld, old_values_n, returns_n, mask, rows_per_chunk, chunk_stride, M, e_clip, clip_value, inv_count, d_value,
                          dv_ld};
    double tot[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int m = 0; m < M; ++m) {
        double acc[3] = {0, 0, 0};
        value_loss_thread(a, m, acc);
        for (int i = 0; i < 3; ++i) tot[i] += acc[i];
    }
    for (int i = 0; i < 8; ++i) partial8[i] = tot[i];
    return B200RL_OK;
}
#endif  // B200RL_TEST_HOOKS
