// bf16 tensor-core (tcgen05 / TMEM / TMA-bulk) MLP kernels: the `mixed_precision: True` path.
//
//   fwd  (train)  : per 128-row tile  X -> a1 -> a2 -> a3 -> heads, with the PPO loss forward+backward fused into the
//                   last epilogue (replaces network_builder.py:494-512 + a2c_continuous.py:97-134 + the loss part of
//                   loss.backward()); saves a1/a2/a3 and d_head as bf16 operand tiles.
//   fwd  (rollout): same trunk, epilogue = sample / neglogp / denorm value written into the arena (models.py:329-364).
//   bwd1          : delta chain d_head -> d3 -> d2 -> d1 (dgrad) + weight grads of the head and layer 3 + bias grads.
//   bwd2          : weight grads of layers 2 and 1 (+ bias grad of layer 1).
//
// All GEMMs are tcgen05.mma (M = 128 rows per tile, fp32 accumulators in TMEM) issued by one thread; operands are
// INTERLEAVE shared-memory tiles (tc_common.cuh).  One packed bf16 copy of each weight matrix serves the forward
// (K-major view) and the dgrad (MN-major view); one copy of each activation / delta tile serves the dgrad
// (K-major) and the wgrad (MN-major) MMAs -- no transposes anywhere.  Tiles move global<->shared with
// cp.async.bulk (1-D TMA) + mbarrier transaction counts; weight gradients stay resident in TMEM across all tiles a
// persistent CTA processes and are flushed once per CTA into a [n_cta][P] partial buffer that the deterministic
// split reducer (mlp_simt.cu) sums.
#include "common.cuh"
#include "loss_math.cuh"
#include "tc_common.cuh"

// One translation unit per MLP activation: the activation is a compile-time constant of every kernel here (a run-time switch inside the
// epilogues grew the forward kernel by 35 % and cost ~10 % of its time).  mlp_tc.cu itself is the ELU unit and also holds the
// activation-independent entry points and the dispatcher; mlp_tc_relu.cu / mlp_tc_tanh.cu define B200RL_TC_ACT and include this file,
// which then only emits their three launchers (b200rl_tcimpl_*_act<N>, hidden visibility).
#ifndef B200RL_TC_ACT
#define B200RL_TC_ACT 1          // B200RL_ACT_ELU
#define B200RL_TC_MAIN 1
#endif
#define B200RL_TC_CAT2(a, b) a##b
#define B200RL_TC_CAT(a, b) B200RL_TC_CAT2(a, b)
#define TCIMPL(name) B200RL_TC_CAT(name##_act, B200RL_TC_ACT)

namespace {
constexpr int TC_ACT = B200RL_TC_ACT;

using namespace tc;

constexpr int FWD_THREADS = 512;   // 16 warps: lane-quarter q = warp & 3 (TMEM lanes 32q..32q+31), column slice h = warp >> 2 (4 slices)

// ---- TMA bulk helpers ---------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,"
        "%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// issue only (no wait): lets an epilogue put two 32-column loads in flight before the first use (tmem_ld_wait() once)
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,"
        "%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float elu_fast(float x) { return x > 0.f ? x : (__expf(x) - 1.0f); }
__device__ __forceinline__ float elu_grad_from_out(float a) { return a > 0.f ? 1.f : a + 1.f; }
__device__ __forceinline__ float tanh_fast(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// v[j] = act(v[j] + bias[j]) over NV accumulator columns; the activation (B200RL_ACT_*) is this translation unit's compile-time constant
// (network_builder.py:132 _build_mlp: one activation for the whole MLP; elu / relu / tanh are what the shipped configs use)
template <int NV>
__device__ __forceinline__ void bias_act(float (&v)[NV], const float* __restrict__ bias) {
    constexpr int act = TC_ACT;
    if (act == B200RL_ACT_ELU) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = elu_fast(v[j] + bias[j]);
    } else if (act == B200RL_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = fmaxf(v[j] + bias[j], 0.f);
    } else if (act == B200RL_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = tanh_fast(v[j] + bias[j]);
    } else {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = v[j] + bias[j];
    }
}
// v[j] *= act'(.) expressed through the activation OUTPUT a[j] (8 bf16 values of one chunk)
__device__ __forceinline__ void mul_act_grad8(float* v, const float (&a)[8]) {
    constexpr int act = TC_ACT;
    if (act == B200RL_ACT_ELU) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] *= elu_grad_from_out(a[j]);
    } else if (act == B200RL_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = a[j] > 0.f ? v[j] : 0.f;
    } else if (act == B200RL_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] *= 1.0f - a[j] * a[j];
    }
}
__device__ __forceinline__ void unpack8_bf16(const uint4& u, float* f) {
    const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 t = __bfloat1622float2(p[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}

// ---- network geometry (compile time) ------------------------------------------------------------------------
// activation-like tiles: 128 rows, C cols: CS = 2048 (col-group stride), RS = 128 (row-group stride), C*256 bytes
// weight tiles [R rows(out) x C cols(in)]: CS = (R/8)*128, RS = 128
template <int DPAD_, int U1_, int U2_, int U3_, int AP_>
struct Net {
    static constexpr int DPAD = DPAD_, U1 = U1_, U2 = U2_, U3 = U3_, AP = AP_;
    static constexpr uint32_t ACS = 2048, ARS = 128;
    static constexpr uint32_t W1_CS = (U1 / 8) * 128, W2_CS = (U2 / 8) * 128, W3_CS = (U3 / 8) * 128, WH_CS = (AP / 8) * 128;
    static constexpr uint32_t W1_BYTES = U1 * DPAD * 2, W2_BYTES = U2 * U1 * 2, W3_BYTES = U3 * U2 * 2, WH_BYTES = AP * U3 * 2;
    static constexpr uint32_t W1_OFF = 0, W2_OFF = W1_BYTES, W3_OFF = W2_OFF + W2_BYTES, WH_OFF = W3_OFF + W3_BYTES;
    static constexpr uint32_t PACK_BYTES = WH_OFF + WH_BYTES;
    static constexpr uint32_t X_BYTES = DPAD * 256, A1_BYTES = U1 * 256, A2_BYTES = U2 * 256, A3_BYTES = U3 * 256, DH_BYTES = AP * 256;
    static_assert(U2 == 128, "wgrad tiles assume a 128-wide second hidden layer (M = 128 MMAs)");
    static_assert(U1 % 128 == 0 && (U1 / 4) % 32 == 0 && (U2 / 4) % 32 == 0, "epilogue column slices are multiples of 32");
    static_assert(U1 % 128 == 0 && U1 <= 256 && U3 <= 128 && U3 % 16 == 0 && DPAD % 16 == 0 && DPAD <= 256 && AP == 16, "unsupported net");
};
using NetC2 = Net<64, 256, 128, 64, 16>;
// Wide observations (64 < D <= 256, e.g. BASELINE configs[4] obs = 256): same hidden layers; layer 1 does not fit beside the other
// weights in one CTA's shared memory (W1 alone is 128 KB), so it runs in kernels of its own (l1_fwd_tc_kernel, l1_wgrad_tc_kernel)
// and the chain kernels are instantiated with XL1 = true ("external layer 1": a1 tiles come from / dW1 goes to those kernels).
using NetW = Net<256, 256, 128, 64, 16>;

// ---- weight packing: fp32 [R, C] row-major -> bf16 INTERLEAVE tile [Rpad, Cpad] ------------------------------
struct PackSeg { const float* src; int R, C, Rpad, Cpad; uint32_t dst_off; };
struct PackArgs { PackSeg seg[4]; };

__global__ void __launch_bounds__(256) pack_weights_kernel(PackArgs a, uint8_t* __restrict__ dst) {
    const PackSeg s = a.seg[blockIdx.y];
    const int ncg = s.Cpad / 8;
    const uint32_t CS = (uint32_t)(s.Rpad / 8) * 128u;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < s.Rpad * ncg; i += gridDim.x * blockDim.x) {
        const int r = i / ncg, cg = i - r * ncg;
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = cg * 8 + j;
            f[j] = (r < s.R && c < s.C) ? __ldg(s.src + (size_t)r * s.C + c) : 0.f;
        }
        *reinterpret_cast<uint4*>(dst + s.dst_off + tile_off(r, cg, CS, 128u)) = pack8_bf16(f);
    }
}

// ---- X tile: fp32 obs rows -> normalise/clamp -> bf16 operand tile ---------------------------------------------
// sNorm: [2*DPAD] floats in shared memory = (mean, 1/std) per column (identity when normalisation is off).  The bf16
// rounding of the operand hides the 1-ulp difference between (x-m)/std and (x-m)*(1/std).
template <class N>
__device__ __forceinline__ void load_norm_smem(float* sNorm, const float* __restrict__ nm, const float* __restrict__ ns, int D) {
    for (int c = threadIdx.x; c < N::DPAD; c += blockDim.x) {
        sNorm[c] = (nm && c < D) ? __ldg(nm + c) : 0.f;
        sNorm[N::DPAD + c] = (ns && c < D) ? __frcp_rn(__ldg(ns + c)) : 1.f;
    }
}
template <class N, int NTHREADS>
__device__ __forceinline__ void stage_x_tile(uint8_t* sX, const float* __restrict__ obs, int64_t row0, int rows_valid, int D,
                                             const float* __restrict__ sNorm, bool do_norm) {
    constexpr int NCG = N::DPAD / 8;
    constexpr int ITEMS = (128 * NCG + NTHREADS - 1) / NTHREADS;
    const bool vec = (D & 3) == 0;
    float4 va[ITEMS], vb[ITEMS];
    // phase 1: issue every global load of this thread (ITEMS x 32 B) before touching any of them
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
        const int i = threadIdx.x + it * NTHREADS;
        const int cg = i / 128, r = i - cg * 128;      // consecutive threads -> consecutive rows (conflict-free 16B stores)
        const int c0 = cg * 8;
        va[it] = make_float4(0.f, 0.f, 0.f, 0.f); vb[it] = va[it];
        if (i < 128 * NCG && r < rows_valid && c0 < D) {
            const float* src = obs + (row0 + r) * D + c0;
            if (vec) {
                va[it] = __ldg(reinterpret_cast<const float4*>(src));
                if (c0 + 4 < D) vb[it] = __ldg(reinterpret_cast<const float4*>(src) + 1);
            } else {
                float t[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) t[j] = (c0 + j < D) ? __ldg(src + j) : 0.f;
                va[it] = make_float4(t[0], t[1], t[2], t[3]); vb[it] = make_float4(t[4], t[5], t[6], t[7]);
            }
        }
    }
    // phase 2: normalise / clamp / pack / store
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
        const int i = threadIdx.x + it * NTHREADS;
        if (i >= 128 * NCG) break;
        const int cg = i / 128, r = i - cg * 128;
        const int c0 = cg * 8;
        float f[8] = {va[it].x, va[it].y, va[it].z, va[it].w, vb[it].x, vb[it].y, vb[it].z, vb[it].w};
        if (do_norm) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                f[j] = (c0 + j < D && r < rows_valid) ? fminf(fmaxf((f[j] - sNorm[c0 + j]) * sNorm[N::DPAD + c0 + j], -5.0f), 5.0f) : 0.f;
        }
        *reinterpret_cast<uint4*>(sX + tile_off(r, cg, N::ACS, N::ARS)) = pack8_bf16(f);
    }
}

// Column-group pass of the same staging for wide tiles: col-groups [cg_base, cg_base + NCGP) of a 128-row tile, so that the loads
// in flight per thread stay bounded (NCGP * 128 / NTHREADS items of 32 B) whatever DPAD is.
template <class N, int NTHREADS, int NCGP>
__host__ __device__ __forceinline__ void stage_x_cols(uint8_t* sX, const float* __restrict__ obs, int64_t row0, int rows_valid, int D,
                                                      const float* __restrict__ sNorm, bool do_norm, int cg_base, int tid) {
    // __host__ __device__ (tid passed in): the index arithmetic is exercised on the CPU by b200rl_hosttest_stage_x_cols
    constexpr int ITEMS = (128 * NCGP + NTHREADS - 1) / NTHREADS;
    static_assert((128 * NCGP) % NTHREADS == 0, "whole passes only");
    const bool vec = (D & 3) == 0;
    float4 va[ITEMS], vb[ITEMS];
#ifdef __CUDA_ARCH__
#define B200RL_LD(p) __ldg(p)
#else
#define B200RL_LD(p) (*(p))
#endif
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
        const int i = tid + it * NTHREADS;
        const int cgl = i / 128, r = i - cgl * 128;
        const int c0 = (cg_base + cgl) * 8;
        va[it] = make_float4(0.f, 0.f, 0.f, 0.f); vb[it] = va[it];
        if (r < rows_valid && c0 < D) {
            const float* src = obs + (row0 + r) * D + c0;
            if (vec) {
                va[it] = B200RL_LD(reinterpret_cast<const float4*>(src));
                if (c0 + 4 < D) vb[it] = B200RL_LD(reinterpret_cast<const float4*>(src) + 1);
            } else {
                float t[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) t[j] = (c0 + j < D) ? B200RL_LD(src + j) : 0.f;
                va[it] = make_float4(t[0], t[1], t[2], t[3]); vb[it] = make_float4(t[4], t[5], t[6], t[7]);
            }
        }
    }
#undef B200RL_LD
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
        const int i = tid + it * NTHREADS;
        const int cgl = i / 128, r = i - cgl * 128;
        const int cg = cg_base + cgl, c0 = cg * 8;
        float f[8] = {va[it].x, va[it].y, va[it].z, va[it].w, vb[it].x, vb[it].y, vb[it].z, vb[it].w};
        if (do_norm) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                f[j] = (c0 + j < D && r < rows_valid) ? fminf(fmaxf((f[j] - sNorm[c0 + j]) * sNorm[N::DPAD + c0 + j], -5.0f), 5.0f) : 0.f;
        }
        *reinterpret_cast<uint4*>(sX + tile_off(r, cg, N::ACS, N::ARS)) = pack8_bf16(f);
    }
}

// Same tile, sourced from a raw fp32 copy of the rows that a 1-D TMA bulk copy (cp.async.bulk) dropped into shared memory
// while the previous tile was still computing: sRaw[r * D + c].  Requires D % 4 == 0.  Quarter-warps read 8 consecutive
// rows x 16 B (row stride D*4 bytes: conflict-free for D = 60) and write 8 consecutive 16 B chunks.
template <class N, int NTHREADS>
__device__ __forceinline__ void stage_x_tile_smem(uint8_t* sX, const float* sRaw, int rows_valid, int D, const float* __restrict__ sNorm,
                                                  bool do_norm) {
    constexpr int NCG = N::DPAD / 8;
#pragma unroll
    for (int it = 0; it < (128 * NCG + NTHREADS - 1) / NTHREADS; ++it) {
        const int i = threadIdx.x + it * NTHREADS;
        if (i >= 128 * NCG) break;
        const int cg = i / 128, r = i - cg * 128;
        const int c0 = cg * 8;
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
        if (r < rows_valid && c0 < D) {
            const float4* src = reinterpret_cast<const float4*>(sRaw + r * D + c0);
            va = src[0];
            if (c0 + 4 < D) vb = src[1];
        }
        float f[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
        if (do_norm) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                f[j] = (c0 + j < D && r < rows_valid) ? fminf(fmaxf((f[j] - sNorm[c0 + j]) * sNorm[N::DPAD + c0 + j], -5.0f), 5.0f) : 0.f;
        }
        *reinterpret_cast<uint4*>(sX + tile_off(r, cg, N::ACS, N::ARS)) = pack8_bf16(f);
    }
}

// Column sums of a bf16 operand tile (bias gradients): R rows, G column groups of 8 columns, column-group stride CS bytes
// (chunk (g, r) sits at g * CS + r * 16).  Thread (g, rs) = (tid / RS, tid % RS) adds rows rs, rs + RS, ... of its 8 columns
// (a quarter-warp reads 8 consecutive 16 B chunks: conflict-free), the RS partials are combined with warp shuffles in a fixed
// order, and the lane with rs == 0 accumulates the result into its 8 running sums.  Whole warps either take part or skip.
template <int R, int G, uint32_t CS, int T>
__device__ __forceinline__ void colsum8(const uint8_t* sT, int tid, float (&acc)[8]) {
    constexpr int RS = (T / G) < 32 ? (T / G) : 32;
    static_assert((RS & (RS - 1)) == 0 && RS >= 1 && RS * G <= T && (RS * G) % 32 == 0, "colsum8 thread mapping");
    const int rs = tid % RS, g = tid / RS;
    if (g >= G) return;
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int r = rs; r < R; r += RS) {
        float a[8];
        unpack8_bf16(*reinterpret_cast<const uint4*>(sT + g * CS + r * 16), a);
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] += a[j];
    }
#pragma unroll
    for (int o = RS / 2; o > 0; o >>= 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
    }
    if (rs == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += s[j];
    }
}
// the thread that owns column group g after colsum8<.., G, .., T> (rs == 0), or -1
template <int G, int T>
__device__ __forceinline__ int colsum8_owner_group(int tid) {
    constexpr int RS = (T / G) < 32 ? (T / G) : 32;
    return (tid % RS == 0 && tid / RS < G) ? tid / RS : -1;
}

// epilogue helper: thread (row r) processes 32 accumulator columns [c0, c0+32): v = elu(v + bias) -> bf16 chunks into
// a shared operand tile and (optionally) the global tiled activation buffer
__device__ __forceinline__ void store_chunks32(const float (&v)[32], int r, int c0, uint8_t* s_tile, uint8_t* g_tile) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 u = pack8_bf16(&v[q * 8]);
        const uint32_t off = tile_off(r, c0 / 8 + q, 2048u, 128u);
        if (s_tile) *reinterpret_cast<uint4*>(s_tile + off) = u;
        if (g_tile) *reinterpret_cast<uint4*>(g_tile + off) = u;
    }
}

// head[1 + h + 4k] without dynamic register-array indexing (h is a runtime warp-group id, k an unrolled constant)
__device__ __forceinline__ float pick_mu(const float (&head)[16], int h, int k) {
    float v = 0.f;
#pragma unroll
    for (int hh = 0; hh < 4; ++hh) {
        const int idx = 1 + hh + 4 * k;
        if (idx < 16 && h == hh) v = head[idx];
    }
    return v;
}

struct FwdArgs {
    const float* obs; int rows_per_chunk; int64_t chunk_stride; int D;
    const float* nm; const float* ns;
    const uint8_t* wpack; const float* b1; const float* b2; const float* b3; const float* bh; const float* logstd;
    int M; int A;
    int u1, u2, u3, act;      // LOGICAL layer widths (<= the compiled Net widths: the packed weights are zero-padded) and B200RL_ACT_*
    // training epilogue
    LossArena la; const float* inv_count_dev; LossCfgDev cfg;
    uint8_t* act1; uint8_t* act2; uint8_t* act3; uint8_t* dhead; double* partials;
    uint8_t* xt;      // optional: normalised bf16 observation tiles for the pipelined backward-2 kernel
    // rollout epilogue
    const double* vms_mean; const double* vms_var; int normalize_value; const float* noise; uint64_t seed;
    const uint64_t* rng_epoch; uint32_t step_index;
    float* actions; float* mus; float* sigmas; float* neglogp; float* values; float* env_actions; int clip_actions;
    const float* act_low; const float* act_high; const uint8_t* dones_cur; uint8_t* dones_out; const float* prev_dones;
    float* valid_out; int values_only;
};

constexpr int LOSS_SLOTS = LOSS_NSC + 32;   // partial row stride shared with loss.cu (NSC + MAXA)

// ================================================================================================= forward
// Opt-in stage timing (tools/tc_stage_timing.py builds a variant with -DB200RL_TC_TIMING): thread 0 of CTA 0 stamps
// clock64() at every stage boundary of its tiles.  Never compiled into the product library.
#ifdef B200RL_TC_TIMING
__device__ long long g_tc_stamp[3 * 128];   // [0,128) fwd, [128,256) bwd1, [256,384) bwd2
#define TSTAMP() do { if (blockIdx.x == 0 && tid == 0 && n_stamp < 127) g_tc_stamp[TSB + 1 + n_stamp++] = clock64(); } while (0)
#define TSTAMP_END() do { if (blockIdx.x == 0 && tid == 0) g_tc_stamp[TSB] = n_stamp; } while (0)
#ifdef B200RL_TC_MAIN
extern "C" B200RL_EXPORT int b200rl_debug_tc_stamps(long long* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, g_tc_stamp, sizeof(long long) * 3 * 128);
}
#endif
#else
#define TSTAMP() do {} while (0)
#define TSTAMP_END() do {} while (0)
#endif

// XL1 ("external layer 1", wide observations): layer 1 ran in l1_fwd_tc_kernel; this kernel TMA-loads the a1 tile from p.act1
// instead of staging X / multiplying by W1 (which is not resident), a3 gets a region of its own so that the NEXT tile's a1 can
// be prefetched as soon as the layer-2 MMAs have read the current one.  XL1 = false compiles to exactly the code it always was.
template <class N, bool TRAIN, bool XL1 = false>
__global__ void __launch_bounds__(FWD_THREADS, 1) mlp_fwd_tc_kernel(const FwdArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr uint32_t SW2 = XL1 ? 0u : N::W2_OFF, SW3 = SW2 + N::W2_BYTES, SWH = SW3 + N::W3_BYTES, SPACK = SWH + N::WH_BYTES;
    static_assert(XL1 || (SW3 == N::W3_OFF && SWH == N::WH_OFF && SPACK == N::PACK_BYTES), "resident-W1 layout unchanged");
    constexpr uint32_t XA2_BYTES = XL1 ? N::A2_BYTES : (N::A2_BYTES > N::X_BYTES ? N::A2_BYTES : N::X_BYTES);
    uint8_t* sW1 = smem + N::W1_OFF; uint8_t* sW2 = smem + SW2; uint8_t* sW3 = smem + SW3; uint8_t* sWh = smem + SWH;
    uint8_t* sA1 = smem + SPACK;                         // a1 (then a3 aliases its start)
    uint8_t* sXA2 = sA1 + N::A1_BYTES;                   // X tile, later a2
    uint8_t* sA3 = XL1 ? sXA2 + XA2_BYTES : sA1;
    // raw fp32 rows of the NEXT tile (TMA prefetch): the part of the a1 region that a3 does not alias; free once MMA 2 has read a1
    float* sXraw = reinterpret_cast<float*>(sA1 + N::A3_BYTES);
    static_assert(XL1 || N::A3_BYTES + 128 * N::DPAD * 4 <= N::A1_BYTES, "X prefetch buffer must fit behind a3 inside the a1 region");
    float* sBias = reinterpret_cast<float*>(sXA2 + XA2_BYTES + (XL1 ? N::A3_BYTES : 0u));
    float* sB1 = sBias; float* sB2 = sB1 + N::U1; float* sB3 = sB2 + N::U2; float* sBh = sB3 + N::U3;
    float* sSig = sBh + N::AP;                           // sigma, logstd, 1/sigma, log(sigma): 4*A floats, then sum(logstd), entropy
    float* sNorm = sSig + 64;                            // [2*DPAD] obs mean, 1/std
    float* sRed = sNorm + 2 * N::DPAD;                   // [4 warps][LOSS_SLOTS] (only the h == 0 warps run the loss)
    double* sAcc = reinterpret_cast<double*>(sRed + 4 * LOSS_SLOTS);     // [LOSS_SLOTS] per-CTA running partial
    uint64_t* bars = reinterpret_cast<uint64_t*>(sAcc + LOSS_SLOTS);     // [0]=W1, [1..4]=mma stages, [5]=X prefetch, [6]=W2, [7]=W3+Wh
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    const int n_tiles = (p.M + 127) / 128;
    int n_stamp = 0; (void)n_stamp;
    constexpr int TSB = 0; (void)TSB;
    TSTAMP();   // kernel start

    // ---- prologue, part 1: nothing here depends on the predecessor kernel (PDL: may overlap its tail) ----
    const bool x_tma = !XL1 && (p.D & 3) == 0;         // 16-byte granularity of the bulk copy
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (tid == 0) {
        for (int i = 0; i < 8; ++i) mbar_init(&bars[i], 1);
        fence_mbar_init();
        if (x_tma && (int)blockIdx.x < n_tiles) {     // observation rows come from the environment, not from the kernel chain
            const int m0 = blockIdx.x * 128;
            const uint32_t bytes = (uint32_t)min(128, p.M - m0) * p.D * 4u;
            mbar_expect_tx(&bars[5], bytes);
            bulk_g2s(sXraw, p.obs + chunk_row(m0, p.rows_per_chunk, p.chunk_stride) * p.D, bytes, &bars[5]);
        }
    }
    TSTAMP();   // TMEM allocated (warp 0), barriers initialised, first X tile requested
    pdl_sync();
    // ---- prologue, part 2: parameters and normaliser statistics (written by the optimiser kernel) ----
    if (tid == 0) {
        if constexpr (XL1) {
            if ((int)blockIdx.x < n_tiles) {      // first a1 tile (written by the predecessor kernel: after pdl_sync)
                mbar_expect_tx(&bars[5], N::A1_BYTES);
                bulk_g2s(sA1, p.act1 + (size_t)blockIdx.x * N::A1_BYTES, N::A1_BYTES, &bars[5]);
            }
        } else {
        // one barrier per consumer so that layer 1 starts as soon as W1 (32 KB of the 114 KB) has landed
        mbar_expect_tx(&bars[0], N::W1_BYTES);
        bulk_g2s(sW1, p.wpack + N::W1_OFF, N::W1_BYTES, &bars[0]);
        }
        mbar_expect_tx(&bars[6], N::W2_BYTES);
        bulk_g2s(sW2, p.wpack + N::W2_OFF, N::W2_BYTES, &bars[6]);
        mbar_expect_tx(&bars[7], N::W3_BYTES + N::WH_BYTES);
        bulk_g2s(sW3, p.wpack + N::W3_OFF, N::W3_BYTES, &bars[7]);
        bulk_g2s(sWh, p.wpack + N::WH_OFF, N::WH_BYTES, &bars[7]);
    }
    // every global load of the prologue lands in a register first -- ONE memory round trip (measured: 2.6 -> 1.6 us for this stretch and
    // 1.1 -> 0.3 us after the barrier, forward+loss 35.8-36.9 -> 33.8 us per launch: profiles/r02_fwd_ab.md) -- then the shared-memory stores
    {
        static_assert(N::U1 <= FWD_THREADS && N::DPAD <= FWD_THREADS, "one element per thread");
        const float r1 = (tid < N::U1 && tid < p.u1) ? __ldg(p.b1 + tid) : 0.f;
        const float r2 = (tid < N::U2 && tid < p.u2) ? __ldg(p.b2 + tid) : 0.f;
        const float r3 = (tid < N::U3 && tid < p.u3) ? __ldg(p.b3 + tid) : 0.f;
        const float rh = (tid < N::AP && tid < p.A + 1) ? __ldg(p.bh + tid) : 0.f;
        const float rl = tid < p.A ? __ldg(p.logstd + tid) : 0.f;
        const float rm = (p.nm && tid < p.D) ? __ldg(p.nm + tid) : 0.f;
        const float rs = (p.ns && tid < p.D) ? __ldg(p.ns + tid) : 1.f;
        if (tid < N::U1) sB1[tid] = r1;
        if (tid < N::U2) sB2[tid] = r2;
        if (tid < N::U3) sB3[tid] = r3;
        if (tid < N::AP) sBh[tid] = rh;
        if (tid < N::DPAD) { sNorm[tid] = rm; sNorm[N::DPAD + tid] = (p.ns && tid < p.D) ? __frcp_rn(rs) : 1.f; }
        if (tid < p.A) { const float sg = expf(rl); sSig[tid] = sg; sSig[p.A + tid] = rl; sSig[2 * p.A + tid] = 1.0f / sg; sSig[3 * p.A + tid] = logf(sg); }
    }
    TSTAMP();   // weight copies issued, parameter loads done
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    TSTAMP();   // the prologue barrier passed
    if (tid == 0) {      // row-independent constants: sum(logstd) and the entropy of the diagonal Gaussian (first reader: the loss epilogue)
        float sl = 0.f, en = 0.f;
        for (int j = 0; j < p.A; ++j) { sl += sSig[p.A + j]; en += 0.5f + 0.9189385332046727f + sSig[3 * p.A + j]; }
        sSig[4 * p.A] = sl; sSig[4 * p.A + 1] = en;
    }
    TSTAMP();   // prologue done
    const uint32_t tmem = *tmem_slot;
    const uint32_t T1 = tmem, T2 = tmem + 256, T3 = tmem + 384, T4 = tmem + 448;     // accumulator column bases
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t phase = 0;
    bool weights_ready = false;
    // per-thread running loss partials over this CTA's tiles (reduced once, after the tile loop): scalars in the h == 0 threads,
    // d_logstd slices (actions h, h+4, h+8, h+12) in every thread
    float sc[LOSS_NSC];
    float dls[4];
#pragma unroll
    for (int i = 0; i < LOSS_NSC; ++i) sc[i] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) dls[k] = 0.f;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int m0 = tile * 128;
        const int rows_valid = min(128, p.M - m0);
        const int64_t arow0 = chunk_row(m0, p.rows_per_chunk, p.chunk_stride);   // tile lies inside one chunk (host-checked)
        TSTAMP();   // tile start
        if constexpr (XL1) {
            mbar_wait(&bars[5], phase);       // a1 tile landed (async-proxy write, async-proxy reader: no generic-proxy fence needed)
            weights_ready = true;
        } else {
        if (x_tma) {
            mbar_wait(&bars[5], phase);
            stage_x_tile_smem<N, FWD_THREADS>(sXA2, sXraw, rows_valid, p.D, sNorm, p.nm != nullptr);
        } else {
            stage_x_tile<N, FWD_THREADS>(sXA2, p.obs, arow0, rows_valid, p.D, sNorm, p.nm != nullptr);
        }
        fence_async_smem();
        if (!weights_ready) { mbar_wait(&bars[0], 0); weights_ready = true; }
        __syncthreads();
        TSTAMP();   // X staged
        if (TRAIN && p.xt) {      // keep the normalised bf16 tile for the weight-gradient kernel (16 B per thread-iteration, coalesced)
            uint4* gx = reinterpret_cast<uint4*>(p.xt + (size_t)tile * N::X_BYTES);
            for (int i = tid; i < (int)N::X_BYTES / 16; i += FWD_THREADS) gx[i] = reinterpret_cast<const uint4*>(sXA2)[i];
        }
        // ---------------- layer 1: T1[128, U1] = X . W1^T ----------------
        if (tid == 0) {
            fence_after_sync();
            constexpr uint32_t idesc = make_idesc_bf16(128, N::U1, 0, 0);
#pragma unroll
            for (int k = 0; k < N::DPAD / 16; ++k)
                umma_bf16(T1, make_smem_desc(smem_u32(sXA2) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sW1) + k * 2 * N::W1_CS, N::W1_CS, 128), idesc, k > 0);
            umma_commit(&bars[1]);
        }
        mbar_wait(&bars[1], phase);
        fence_after_sync();
        TSTAMP();   // MMA 1 done
        {
            uint8_t* g1 = TRAIN ? p.act1 + (size_t)tile * N::A1_BYTES : nullptr;
#pragma unroll 1
            for (int c0 = h * (N::U1 / 4); c0 < (h + 1) * (N::U1 / 4); c0 += 32) {
                float v[32];
                tmem_ld32(T1 + lane_base + c0, v);
                bias_act<32>(v, sB1 + c0);
                store_chunks32(v, row, c0, sA1, g1);
            }
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        }   // !XL1
        TSTAMP();   // epilogue 1 done
        // ---------------- layer 2: T2[128, U2] = a1 . W2^T ----------------
        if (tid == 0) {
            if (tile == (int)blockIdx.x) mbar_wait(&bars[6], 0);       // W2 landed (first tile only)
            fence_after_sync();
            constexpr uint32_t idesc = make_idesc_bf16(128, N::U2, 0, 0);
#pragma unroll
            for (int k = 0; k < N::U1 / 16; ++k)
                umma_bf16(T2, make_smem_desc(smem_u32(sA1) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sW2) + k * 2 * N::W2_CS, N::W2_CS, 128), idesc, k > 0);
            umma_commit(&bars[2]);
        }
        mbar_wait(&bars[2], phase);
        fence_after_sync();
        TSTAMP();   // MMA 2 done
        if (XL1 && tid == 0 && tile + (int)gridDim.x < n_tiles) {
            // a1 is dead now: fetch the next tile's a1 (a3 has its own region in this layout)
            mbar_expect_tx(&bars[5], N::A1_BYTES);
            bulk_g2s(sA1, p.act1 + (size_t)(tile + gridDim.x) * N::A1_BYTES, N::A1_BYTES, &bars[5]);
        }
        if (tid == 0 && x_tma && tile + (int)gridDim.x < n_tiles) {
            // a1 is dead now (its readers, the layer-2 MMAs, have completed): prefetch the next tile's rows behind a3
            const int m1 = (tile + gridDim.x) * 128;
            const uint32_t bytes = (uint32_t)min(128, p.M - m1) * p.D * 4u;
            mbar_expect_tx(&bars[5], bytes);
            bulk_g2s(sXraw, p.obs + chunk_row(m1, p.rows_per_chunk, p.chunk_stride) * p.D, bytes, &bars[5]);
        }
        {
            uint8_t* g2 = TRAIN ? p.act2 + (size_t)tile * N::A2_BYTES : nullptr;
#pragma unroll 1
            for (int c0 = h * (N::U2 / 4); c0 < (h + 1) * (N::U2 / 4); c0 += 32) {
                float v[32];
                tmem_ld32(T2 + lane_base + c0, v);
                bias_act<32>(v, sB2 + c0);
                store_chunks32(v, row, c0, sXA2, g2);
            }
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        TSTAMP();   // epilogue 2 done
        // ---------------- layer 3: T3[128, U3] = a2 . W3^T ----------------
        if (tid == 0) {
            if (tile == (int)blockIdx.x) mbar_wait(&bars[7], 0);       // W3 and the head weights landed (first tile only)
            fence_after_sync();
            constexpr uint32_t idesc = make_idesc_bf16(128, N::U3, 0, 0);
#pragma unroll
            for (int k = 0; k < N::U2 / 16; ++k)
                umma_bf16(T3, make_smem_desc(smem_u32(sXA2) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sW3) + k * 2 * N::W3_CS, N::W3_CS, 128), idesc, k > 0);
            umma_commit(&bars[3]);
        }
        mbar_wait(&bars[3], phase);
        fence_after_sync();
        TSTAMP();   // MMA 3 done
        {
            uint8_t* g3 = TRAIN ? p.act3 + (size_t)tile * N::A3_BYTES : nullptr;
            // U3/4 = 16 columns per thread
            static_assert(N::U3 / 4 == 16, "layer-3 epilogue assumes 16 columns per column slice");
            const int c0 = h * 16;
            float v[16];
            tmem_ld16(T3 + lane_base + c0, v);
            bias_act<16>(v, sB3 + c0);
#pragma unroll
            for (int qq = 0; qq < 2; ++qq) {
                const uint4 u = pack8_bf16(&v[qq * 8]);
                const uint32_t off = tile_off(row, c0 / 8 + qq, 2048u, 128u);
                *reinterpret_cast<uint4*>(sA3 + off) = u;
                if (g3) *reinterpret_cast<uint4*>(g3 + off) = u;
            }
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        TSTAMP();   // epilogue 3 done
        // ---------------- heads: T4[128, AP] = a3 . Wh^T ----------------
        if (tid == 0) {
            fence_after_sync();
            constexpr uint32_t idesc = make_idesc_bf16(128, N::AP, 0, 0);
#pragma unroll
            for (int k = 0; k < N::U3 / 16; ++k)
                umma_bf16(T4, make_smem_desc(smem_u32(sA3) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sWh) + k * 2 * N::WH_CS, N::WH_CS, 128), idesc, k > 0);
            umma_commit(&bars[4]);
        }
        if (TRAIN) {
            // ---- PPO loss, split 4 ways: the four threads (h = 0..3) that can read TMEM lane `row` each take the actions
            //      j = h, h+4, h+8, h+12; per-row sums are exchanged through shared memory (the dead a2 tile region).
            const bool live = row < rows_valid;
            const int64_t ar = arow0 + row;
            float act[4], omu[4], osg[4];
            float old_v = 0.f, ret = 0.f, old_nlp = 0.f, adv = 0.f, mk = 0.f;
            if (live) {      // arena inputs: issued before the wait on the heads MMA so their latency overlaps with it
                old_v = __ldg(p.la.old_values_n + ar); ret = __ldg(p.la.returns_n + ar);
                old_nlp = __ldg(p.la.old_neglogp + ar); adv = __ldg(p.la.advs_n + ar);
                mk = p.la.mask ? __ldg(p.la.mask + ar) : 1.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int j = h + 4 * k;
                    if (j < p.A) { act[k] = __ldg(p.la.actions + ar * p.A + j); omu[k] = p.la.old_mu[ar * p.A + j]; osg[k] = p.la.old_sigma[ar * p.A + j]; }
                }
            }
            mbar_wait(&bars[4], phase);
            fence_after_sync();
            TSTAMP();   // MMA 4 done
            float head[16];
            tmem_ld16(T4 + lane_base, head);
#pragma unroll
            for (int j = 0; j < 16; ++j) head[j] += sBh[j];
            float* sPart = reinterpret_cast<float*>(sXA2);           // [128 rows][4 h][4]: sum z^2, kl, bound loss
            float z[4];
            {
                float sz2 = 0.f, kl = 0.f, bl = 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int j = h + 4 * k;
                    z[k] = 0.f;
                    if (live && j < p.A) {
                        const float mu = pick_mu(head, h, k), sg = sSig[j], isg = sSig[2 * p.A + j];
                        z[k] = (act[k] - mu) * isg;
                        sz2 += z[k] * z[k];
                        const float c1 = __logf(osg[k] * isg + 1e-5f);
                        const float dm = omu[k] - mu;
                        kl += c1 + (sg * sg + dm * dm) * __frcp_rn(2.0f * (osg[k] * osg[k] + 1e-5f)) - 0.5f;
                        if (p.cfg.has_bounds) {
                            if (p.cfg.bound_type == 1) { const float hi = fmaxf(mu - 1.1f, 0.f), lo = fminf(mu + 1.1f, 0.f); bl += lo * lo + hi * hi; }
                            else if (p.cfg.bound_type == 2) bl += mu * mu;
                        }
                    }
                }
                *reinterpret_cast<float4*>(sPart + (row * 4 + h) * 4) = make_float4(sz2, kl, bl, 0.f);
            }
            uint8_t* gd = p.dhead + (size_t)tile * N::DH_BYTES;
            if (live && h >= 2 && p.A + 1 < 8 * (h - 1)) {
                // d_head columns past the last action: the backward MMAs contract over all AP columns of the tile, and a zero weight row
                // cancels stale finite data but not NaN / Inf left in a buffer that was never initialised.  One 16-byte store zeroes
                // each 8-column chunk that holds such columns (h == 2: columns 0-7, h == 3: 8-15); the live columns of the chunk are
                // stored over it after the barrier.
                *reinterpret_cast<uint4*>(gd + tile_off(row, h - 2, 2048u, 128u)) = make_uint4(0, 0, 0, 0);
            }
            __syncthreads();
            TSTAMP();   // loss phase A done
            if (live) {
                float sz2 = 0.f, kl = 0.f, bl = 0.f;
#pragma unroll
                for (int hh = 0; hh < 4; ++hh) { const float4 t4 = *reinterpret_cast<const float4*>(sPart + (row * 4 + hh) * 4); sz2 += t4.x; kl += t4.y; bl += t4.z; }
                const float nlp = 0.5f * sz2 + 0.9189385332046727f * (float)p.A + sSig[4 * p.A];     // sSig[4A] = sum(logstd), [4A+1] = entropy
                const float inv_cnt = p.inv_count_dev ? __ldg(p.inv_count_dev) : (1.0f / (float)p.M);
                const float w = mk * inv_cnt;
                float a_loss, g_a;
                if (p.cfg.ppo) {
                    const float ratio = __expf(old_nlp - nlp);
                    const float mi = 1.0f - p.cfg.e_clip, mx = 1.0f + p.cfg.e_clip;
                    float clamped, dcl;
                    if (p.cfg.smooth) {
                        const float sg_ = __frcp_rn(1.0f + __expf((-(ratio - mi) * __frcp_rn(mx - mi) + 0.5f) * 4.0f));
                        clamped = sg_ * (mx - mi) + mi; dcl = 4.0f * sg_ * (1.0f - sg_);
                    } else {
                        clamped = fminf(fmaxf(ratio, mi), mx); dcl = (ratio >= mi && ratio <= mx) ? 1.0f : 0.0f;
                    }
                    const float t1 = -(adv * ratio), t2 = -(adv * clamped);
                    a_loss = fmaxf(t1, t2);
                    const float d1 = adv * ratio, d2 = adv * dcl * ratio;
                    g_a = (t1 > t2) ? d1 : ((t1 < t2) ? d2 : 0.5f * (d1 + d2));
                } else { a_loss = nlp * adv; g_a = adv; }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int j = h + 4 * k;
                    if (j < p.A) {
                        const float mu = pick_mu(head, h, k), isg = sSig[2 * p.A + j];
                        float db = 0.f;
                        if (p.cfg.has_bounds) {
                            if (p.cfg.bound_type == 1) db = 2.0f * fmaxf(mu - 1.1f, 0.f) + 2.0f * fminf(mu + 1.1f, 0.f);
                            else if (p.cfg.bound_type == 2) db = 2.0f * mu;
                        }
                        const float dmu = w * (g_a * -(z[k] * isg) + p.cfg.bounds_coef * db);
                        dls[k] += w * g_a * (1.0f - z[k] * z[k]);
                        p.la.old_mu[ar * p.A + j] = mu;               // new mu/sigma overwrite the old ones (datasets.py:33-43)
                        p.la.old_sigma[ar * p.A + j] = sSig[j];
                        const int c = 1 + j;
                        *reinterpret_cast<__nv_bfloat16*>(gd + tile_off(row, c >> 3, 2048u, 128u) + (c & 7) * 2) = __float2bfloat16_rn(dmu);
                    }
                }
                if (h == 0) {
                    const float val = head[0];
                    float c_loss, dc;
                    if (p.cfg.clip_value) {
                        const float delta = val - old_v;
                        const float vpc = old_v + fminf(fmaxf(delta, -p.cfg.e_clip), p.cfg.e_clip);
                        const float e1 = val - ret, e2 = vpc - ret;
                        const float l1 = e1 * e1, l2 = e2 * e2;
                        c_loss = fmaxf(l1, l2);
                        const float g1 = 2.0f * e1, g2 = (delta >= -p.cfg.e_clip && delta <= p.cfg.e_clip) ? 2.0f * e2 : 0.0f;
                        dc = (l1 > l2) ? g1 : ((l1 < l2) ? g2 : 0.5f * (g1 + g2));
                    } else { const float e1 = ret - val; c_loss = e1 * e1; dc = -2.0f * e1; }
                    *reinterpret_cast<__nv_bfloat16*>(gd + tile_off(row, 0, 2048u, 128u)) = __float2bfloat16_rn(w * 0.5f * p.cfg.critic_coef * dc);
                    const float lr_ = old_nlp - nlp;
                    const float clipped = (lr_ < p.cfg.log_lo || lr_ > p.cfg.log_hi) ? 1.f : 0.f;
                    sc[0] += w * a_loss; sc[1] += w * c_loss; sc[2] += w * sSig[4 * p.A + 1]; sc[3] += w * bl; sc[4] += w * kl;
                    sc[5] += mk; sc[6] += mk * clipped; sc[7] += w;
                }
            } else if (h < 2) {
                // padded rows of a partial tile: zero d_head so the backward kernels see no contribution
                *reinterpret_cast<uint4*>(gd + tile_off(row, h, 2048u, 128u)) = make_uint4(0, 0, 0, 0);
            }
        } else if (h == 0) {
            mbar_wait(&bars[4], phase);
            fence_after_sync();
            float head[16];
            tmem_ld16(T4 + lane_base, head);
#pragma unroll
            for (int j = 0; j < 16; ++j) head[j] += sBh[j];
            const int m = m0 + row;
            if (row < rows_valid) {
                {
                    // ---- rollout epilogue: models.py:329-364 eval branch ----
                    float val = head[0];
                    if (p.normalize_value) {
                        const float mm = (float)p.vms_mean[0], ss = __fsqrt_rn(__fadd_rn((float)p.vms_var[0], 1e-5f));
                        val = __fadd_rn(__fmul_rn(ss, fminf(fmaxf(val, -5.0f), 5.0f)), mm);
                    }
                    p.values[m] = val;
                    if (!p.values_only) {
                        float eps[16];
                        if (p.noise) {
#pragma unroll
                            for (int j = 0; j < 15; ++j) eps[j] = (j < p.A) ? __ldg(p.noise + (int64_t)m * p.A + j) : 0.f;
                        } else {
                            const uint64_t ep = p.rng_epoch ? *p.rng_epoch : 0ull;
#pragma unroll
                            for (int qq = 0; qq < 4; ++qq) {
                                if (qq * 4 < p.A) {
                                    const Philox4 r4 = philox4x32_10((uint64_t)m, (ep << 20) | ((uint64_t)p.step_index << 4) | (uint64_t)qq, p.seed);
                                    box_muller(r4.x, r4.y, eps[qq * 4 + 0], eps[qq * 4 + 1]);
                                    box_muller(r4.z, r4.w, eps[qq * 4 + 2], eps[qq * 4 + 3]);
                                }
                            }
                        }
                        float sumz2 = 0.f, sumls = 0.f;
                        float av[16], ev[16];
#pragma unroll
                        for (int j = 0; j < 15; ++j) {
                            av[j] = 0.f; ev[j] = 0.f;
                            if (j < p.A) {
                                const float mu = head[1 + j], sg = sSig[j];
                                const float act = __fadd_rn(mu, __fmul_rn(sg, eps[j]));
                                const float z = (act - mu) * sSig[2 * p.A + j];
                                sumz2 += z * z;
                                sumls += sSig[p.A + j];
                                av[j] = act;
                                float ea = act;
                                if (p.env_actions && p.clip_actions) {
                                    const float lo = __ldg(p.act_low + j), hi = __ldg(p.act_high + j);
                                    ea = fminf(fmaxf(act, -1.0f), 1.0f) * ((hi - lo) * 0.5f) + (hi + lo) * 0.5f;
                                }
                                ev[j] = ea;
                            }
                        }
                        av[15] = 0.f; ev[15] = 0.f;
                        // row-wide outputs (A contiguous floats per row in each arena): 16-byte stores when A % 4 == 0
                        if ((p.A & 3) == 0 && ((reinterpret_cast<uintptr_t>(p.actions) | reinterpret_cast<uintptr_t>(p.mus) | reinterpret_cast<uintptr_t>(p.sigmas) |
                                                reinterpret_cast<uintptr_t>(p.env_actions)) & 15) == 0) {
#pragma unroll
                            for (int qq = 0; qq < 4; ++qq) {
                                if (qq * 4 < p.A) {
                                    reinterpret_cast<float4*>(p.actions + (int64_t)m * p.A)[qq] = make_float4(av[qq * 4], av[qq * 4 + 1], av[qq * 4 + 2], av[qq * 4 + 3]);
                                    reinterpret_cast<float4*>(p.mus + (int64_t)m * p.A)[qq] =
                                        make_float4(head[1 + qq * 4], head[2 + qq * 4], head[3 + qq * 4], qq < 3 ? head[(4 + qq * 4) & 15] : 0.f);
                                    reinterpret_cast<float4*>(p.sigmas + (int64_t)m * p.A)[qq] = make_float4(sSig[qq * 4], sSig[qq * 4 + 1], sSig[qq * 4 + 2], sSig[qq * 4 + 3]);
                                    if (p.env_actions)
                                        reinterpret_cast<float4*>(p.env_actions + (int64_t)m * p.A)[qq] = make_float4(ev[qq * 4], ev[qq * 4 + 1], ev[qq * 4 + 2], ev[qq * 4 + 3]);
                                }
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 15; ++j) {
                                if (j < p.A) {
                                    p.actions[(int64_t)m * p.A + j] = av[j];
                                    p.mus[(int64_t)m * p.A + j] = head[1 + j];
                                    p.sigmas[(int64_t)m * p.A + j] = sSig[j];
                                    if (p.env_actions) p.env_actions[(int64_t)m * p.A + j] = ev[j];
                                }
                            }
                        }
                        p.neglogp[m] = 0.5f * sumz2 + 0.9189385332046727f * (float)p.A + sumls;
                        if (p.dones_out) p.dones_out[m] = p.dones_cur[m];
                        if (p.valid_out) p.valid_out[m] = p.prev_dones ? (1.0f - p.prev_dones[m]) : 1.0f;
                    }
                }
            }
        } else {
            mbar_wait(&bars[4], phase);      // rollout: the other column slices only wait for the tile to finish
            fence_after_sync();
        }
        fence_before_sync();
        __syncthreads();
        TSTAMP();   // loss phase B done (tile end)
        phase ^= 1;
    }
    if (!weights_ready) { if (!XL1) mbar_wait(&bars[0], 0); mbar_wait(&bars[6], 0); mbar_wait(&bars[7], 0); }
    if (TRAIN) {
        // block reduction of the loss partials (fixed order => deterministic): scalars from the four h == 0 warps, d_logstd
        // slices from all 16 warps (action j lives in the warps with h == j % 4, slot j / 4)
#pragma unroll
        for (int i = 0; i < LOSS_NSC; ++i) sc[i] = warp_sum(sc[i]);
#pragma unroll
        for (int k = 0; k < 4; ++k) dls[k] = warp_sum(dls[k]);
        if (lane == 0) {
            if (h == 0) {
#pragma unroll
                for (int i = 0; i < LOSS_NSC; ++i) sRed[warp * LOSS_NSC + i] = sc[i];
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) sRed[4 * LOSS_NSC + warp * 4 + k] = dls[k];
        }
    }
    __syncthreads();
    if (TRAIN && tid < LOSS_NSC + p.A) {
        double s = 0.0;
        if (tid < LOSS_NSC) {
            for (int wv = 0; wv < 4; ++wv) s += (double)sRed[wv * LOSS_NSC + tid];
        } else {
            const int j = tid - LOSS_NSC;
            for (int qq = 0; qq < 4; ++qq) s += (double)sRed[4 * LOSS_NSC + (qq + 4 * (j & 3)) * 4 + (j >> 2)];
        }
        p.partials[(int64_t)blockIdx.x * LOSS_SLOTS + tid] = s;
    }
    fence_before_sync();
    __syncthreads();
    TSTAMP();   // kernel end
    TSTAMP_END();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// ================================================================================================= backward 1
struct Bwd1Args {
    const uint8_t* wpack; const uint8_t* act1; const uint8_t* act2; const uint8_t* act3; const uint8_t* dhead;
    uint8_t* delta2; uint8_t* delta1; float* part;   // part: [n_cta][P]
    int M; int A; int P; int off_W3, off_b3, off_b2, off_Wh, off_bh;
    int u1, u2, u3, act;
};

// body: TMEM (512 columns at `tmem`) is allocated by the calling kernel; barriers and shared-memory layout are set up here
template <class N>
__device__ __forceinline__ void bwd1_body(const Bwd1Args& p, uint8_t* smem, const uint32_t tmem) {
    uint8_t* sWh = smem; uint8_t* sW3 = sWh + N::WH_BYTES; uint8_t* sW2 = sW3 + N::W3_BYTES;
    uint8_t* sDH = sW2 + N::W2_BYTES;
    uint8_t* sA3 = sDH + N::DH_BYTES;             // padded to 128 columns (upper col-groups stay zero)
    uint8_t* sA2 = sA3 + 128 * 256;
    uint8_t* sD3 = sA2 + N::A2_BYTES;
    uint8_t* sD2 = sD3 + N::A3_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sD2 + N::A2_BYTES);       // [0] weights, [1] tile loads, [2..4] mma
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    const int n_tiles = (p.M + 127) / 128;
    int n_stamp = 0; (void)n_stamp;
    constexpr int TSB = 128; (void)TSB;
    TSTAMP();   // kernel start
    if (tid == 0) {
        for (int i = 0; i < 5; ++i) mbar_init(&bars[i], 1);
        fence_mbar_init();
    }
    // zero the padding col-groups of the a3 tile once
    for (int i = tid; i < (128 * 256 - (int)N::A3_BYTES) / 16; i += 256) reinterpret_cast<uint4*>(sA3 + N::A3_BYTES)[i] = make_uint4(0, 0, 0, 0);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    pdl_sync();      // everything above is CTA-local; all global traffic comes after the predecessor (the forward kernel) completed
    const uint32_t TT = tmem, TWH = tmem + 256, TW3 = tmem + 288;     // transient [0,256), dWh^T [256,272), dW3^T [288,352)
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    if (tid == 0) {
        mbar_expect_tx(&bars[0], N::WH_BYTES + N::W3_BYTES + N::W2_BYTES);
        bulk_g2s(sWh, p.wpack + N::WH_OFF, N::WH_BYTES, &bars[0]);
        bulk_g2s(sW3, p.wpack + N::W3_OFF, N::W3_BYTES, &bars[0]);
        bulk_g2s(sW2, p.wpack + N::W2_OFF, N::W2_BYTES, &bars[0]);
        if ((int)blockIdx.x < n_tiles) {      // first tile's operands
            const int tile = blockIdx.x;
            mbar_expect_tx(&bars[1], N::DH_BYTES + N::A3_BYTES + N::A2_BYTES);
            bulk_g2s(sDH, p.dhead + (size_t)tile * N::DH_BYTES, N::DH_BYTES, &bars[1]);
            bulk_g2s(sA3, p.act3 + (size_t)tile * N::A3_BYTES, N::A3_BYTES, &bars[1]);
            bulk_g2s(sA2, p.act2 + (size_t)tile * N::A2_BYTES, N::A2_BYTES, &bars[1]);
        }
    }
    // running bias-gradient sums: 8 columns per owning thread (colsum8)
    float bsum3[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, bsum2[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, bsumh[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    uint32_t phase = 0;
    bool first = true;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (first) mbar_wait(&bars[0], 0);
        TSTAMP();   // tile start
        mbar_wait(&bars[1], phase);
        TSTAMP();   // tile loads landed
        // ---- d3pre = d_head . Wh   ;  dWh^T += a3^T . d_head ----
        if (tid == 0) {
            fence_after_sync();
            umma_bf16(TT, make_smem_desc(smem_u32(sDH), N::ACS, N::ARS), make_smem_desc(smem_u32(sWh), 128, N::WH_CS),
                      make_idesc_bf16(128, N::U3, 0, 1), 0);
#pragma unroll
            for (int k = 0; k < 8; ++k)
                umma_bf16(TWH, make_smem_desc(smem_u32(sA3) + k * 256, 128, N::ACS), make_smem_desc(smem_u32(sDH) + k * 256, 128, N::ACS),
                          make_idesc_bf16(128, N::AP, 1, 1), (!first || k > 0) ? 1u : 0u);
            umma_commit(&bars[2]);
        }
        colsum8<128, N::AP / 8, N::ACS, 256>(sDH, tid, bsumh);     // bias grad of the heads
        mbar_wait(&bars[2], phase);
        fence_after_sync();
        TSTAMP();   // MMA a done
        {   // d3 = d3pre * elu'(a3): U3/2 = 32 columns per thread
            const int c0 = h * (N::U3 / 2);
            float v[32];
            tmem_ld32(TT + lane_base + c0, v);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float a[8];
                unpack8_bf16(*reinterpret_cast<const uint4*>(sA3 + tile_off(row, c0 / 8 + g, N::ACS, N::ARS)), a);
                mul_act_grad8(&v[g * 8], a);
            }
            store_chunks32(v, row, c0, sD3, nullptr);
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        TSTAMP();   // d3 epilogue done
        // ---- d2pre = d3 . W3 ; dW3^T += a2^T . d3 ----
        if (tid == 0) {
            fence_after_sync();
#pragma unroll
            for (int k = 0; k < N::U3 / 16; ++k)
                umma_bf16(TT, make_smem_desc(smem_u32(sD3) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sW3) + k * 256, 128, N::W3_CS), make_idesc_bf16(128, N::U2, 0, 1), k > 0);
#pragma unroll
            for (int k = 0; k < 8; ++k)
                umma_bf16(TW3, make_smem_desc(smem_u32(sA2) + k * 256, 128, N::ACS), make_smem_desc(smem_u32(sD3) + k * 256, 128, N::ACS),
                          make_idesc_bf16(128, N::U3, 1, 1), (!first || k > 0) ? 1u : 0u);
            umma_commit(&bars[3]);
        }
        colsum8<128, N::U3 / 8, N::ACS, 256>(sD3, tid, bsum3);
        mbar_wait(&bars[3], phase);
        fence_after_sync();
        TSTAMP();   // MMA b done
        {   // d2 = d2pre * elu'(a2): U2/2 = 64 columns per thread
            uint8_t* g2 = p.delta2 + (size_t)tile * N::A2_BYTES;
#pragma unroll 1
            for (int c0 = h * (N::U2 / 2); c0 < (h + 1) * (N::U2 / 2); c0 += 32) {
                float v[32];
                tmem_ld32(TT + lane_base + c0, v);
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    float a[8];
                    unpack8_bf16(*reinterpret_cast<const uint4*>(sA2 + tile_off(row, c0 / 8 + g, N::ACS, N::ARS)), a);
                    mul_act_grad8(&v[g * 8], a);
                }
                store_chunks32(v, row, c0, sD2, g2);
            }
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        TSTAMP();   // d2 epilogue done
        // ---- d1pre = d2 . W2 ----
        if (tid == 0) {
            fence_after_sync();
            if (tile + (int)gridDim.x < n_tiles) {
                // d_head / a3 / a2 tiles are dead (MMAs a, b completed, epilogue reads fenced + synced): prefetch the next tile's
                // operands so that they land while d1pre and its 128-column epilogue run
                const int nt = tile + gridDim.x;
                mbar_expect_tx(&bars[1], N::DH_BYTES + N::A3_BYTES + N::A2_BYTES);
                bulk_g2s(sDH, p.dhead + (size_t)nt * N::DH_BYTES, N::DH_BYTES, &bars[1]);
                bulk_g2s(sA3, p.act3 + (size_t)nt * N::A3_BYTES, N::A3_BYTES, &bars[1]);
                bulk_g2s(sA2, p.act2 + (size_t)nt * N::A2_BYTES, N::A2_BYTES, &bars[1]);
            }
#pragma unroll
            for (int k = 0; k < N::U2 / 16; ++k)
                umma_bf16(TT, make_smem_desc(smem_u32(sD2) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sW2) + k * 256, 128, N::W2_CS), make_idesc_bf16(128, N::U1, 0, 1), k > 0);
            umma_commit(&bars[4]);
        }
        colsum8<128, N::U2 / 8, N::ACS, 256>(sD2, tid, bsum2);
        mbar_wait(&bars[4], phase);
        fence_after_sync();
        TSTAMP();   // MMA c done
        {   // d1 = d1pre * elu'(a1) straight to the global tiled buffer (a1 read from its global tile, coalesced 16B)
            const uint8_t* ga1 = p.act1 + (size_t)tile * N::A1_BYTES;
            uint8_t* g1 = p.delta1 + (size_t)tile * N::A1_BYTES;
#pragma unroll 1
            for (int c0 = h * (N::U1 / 2); c0 < (h + 1) * (N::U1 / 2); c0 += 32) {
                uint4 ua[4];
#pragma unroll
                for (int g = 0; g < 4; ++g) ua[g] = __ldg(reinterpret_cast<const uint4*>(ga1 + tile_off(row, c0 / 8 + g, N::ACS, N::ARS)));
                float v[32];
                tmem_ld32(TT + lane_base + c0, v);
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    float a[8];
                    unpack8_bf16(ua[g], a);
                    mul_act_grad8(&v[g * 8], a);
                }
                store_chunks32(v, row, c0, nullptr, g1);
            }
        }
        fence_before_sync();
        __syncthreads();
        TSTAMP();   // d1 epilogue done
        phase ^= 1;
        first = false;
    }
    if (first) mbar_wait(&bars[0], 0);
    // ---- flush: dW3^T (TMEM rows = in index, cols = out index), dWh^T, bias sums ----
    float* part = p.part + (size_t)blockIdx.x * p.P;
    const bool native = p.u1 == N::U1 && p.u2 == N::U2 && p.u3 == N::U3;
    fence_after_sync();
    if (!first) {
        {   // dW3^T[i][o] -> grad_W3[o * U2 + i]; thread row = i, cols [32h, 32h+32) of U3 = 64
            const int c0 = h * (N::U3 / 2);
            float v[32];
            tmem_ld32(TW3 + lane_base + c0, v);
            if (native) {          // compile-time strides (immediate offsets): the path of the [256,128,64] geometry
#pragma unroll
                for (int j = 0; j < 32; ++j) part[p.off_W3 + (c0 + j) * N::U2 + row] = v[j];
            } else if (row < p.u2) {
                float* dst = part + p.off_W3 + c0 * p.u2 + row;
                const int nv = p.u3 - c0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < nv) dst[j * p.u2] = v[j];
            }
        }
        if (h == 0) {   // dWh^T[i][o]: rows i < u3 valid; grad_Wh[o * u3 + i], o < A + 1
            // tcgen05.ld is warp-collective (.sync.aligned): every lane of the h == 0 warps executes it, whatever u3 is (a logical width
            // that is not a multiple of 32 must not split a warp around it), only the stores are predicated
            float v[16];
            tmem_ld16(TWH + lane_base, v);
            if (row < p.u3) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (j < p.A + 1) part[p.off_Wh + j * p.u3 + row] = v[j];
            }
        }
    } else {
        for (int i = tid; i < p.u3 * p.u2; i += 256) part[p.off_W3 + i] = 0.f;
        for (int i = tid; i < (p.A + 1) * p.u3; i += 256) part[p.off_Wh + i] = 0.f;
    }
    {
        int g = colsum8_owner_group<N::U3 / 8, 256>(tid);
        if (g >= 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (g * 8 + j < p.u3) part[p.off_b3 + g * 8 + j] = bsum3[j];
        }
        g = colsum8_owner_group<N::U2 / 8, 256>(tid);
        if (g >= 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (g * 8 + j < p.u2) part[p.off_b2 + g * 8 + j] = bsum2[j];
        }
        g = colsum8_owner_group<N::AP / 8, 256>(tid);
        if (g >= 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (g * 8 + j < p.A + 1) part[p.off_bh + g * 8 + j] = bsumh[j];
        }
    }
    fence_before_sync();
    __syncthreads();
    TSTAMP();   // flush done
    TSTAMP_END();
}

// TMEM allocation shared by the backward kernels: warp 0 allocates all 512 columns, every thread learns the base
__device__ __forceinline__ uint32_t bwd_tmem_alloc(uint32_t* slot) {
    if ((threadIdx.x >> 5) == 0) tmem_alloc(slot, 512);
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    return *slot;
}

template <class N>
__global__ void __launch_bounds__(256, 1) mlp_bwd1_tc_kernel(const Bwd1Args p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t tmem_slot;
    const uint32_t tmem = bwd_tmem_alloc(&tmem_slot);
    bwd1_body<N>(p, smem, tmem);
    if ((threadIdx.x >> 5) == 0) tmem_dealloc(tmem, 512);
}

// ================================================================================================= backward 2
struct Bwd2Args {
    const float* obs; int rows_per_chunk; int64_t chunk_stride; int D; const float* nm; const float* ns;
    const uint8_t* act1; const uint8_t* delta2; const uint8_t* delta1; float* part;
    int M; int P; int off_W2, off_W1, off_b1;
    int u1, u2;
    const uint8_t* xt;     // optional (resident-W1 geometry): the normalised bf16 observation tiles the training forward emitted
};

// XL1 (wide observations): dW1 is l1_wgrad_tc_kernel's job -- no X tile, no dW1^T accumulator, no W1 flush here (db1 stays).
template <class N, bool XL1 = false>
__device__ __forceinline__ void bwd2_body(const Bwd2Args& p, uint8_t* smem, const uint32_t tmem) {
    // dW2^T[i][o] = sum_r a1[r][i] d2[r][o]   (two M = 128 halves over i, N = U2)      -> grad_W2[o*U1 + i]
    // dW1^T[i][o] = sum_r x[r][i]  d1[r][o]   (x tile zero-padded to 128 columns, N = U1) -> grad_W1[o*D + i]
    // TMEM lanes carry the contiguous `in` index, so the flush stores are coalesced.
    uint8_t* sD2 = smem; uint8_t* sD1 = sD2 + N::A2_BYTES; uint8_t* sA1 = sD1 + N::A1_BYTES; uint8_t* sX = sA1 + N::A1_BYTES;   // sX: 128 cols
    float* sNorm = reinterpret_cast<float*>(sX + (XL1 ? 0 : 128 * 256));
    uint64_t* bars = reinterpret_cast<uint64_t*>(sNorm + (XL1 ? 0 : 2 * N::DPAD));          // [0] tile loads, [1] mma
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    const int n_tiles = (p.M + 127) / 128;
    int n_stamp = 0; (void)n_stamp;
    constexpr int TSB = 256; (void)TSB;
    TSTAMP();   // kernel start
    if (tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    pdl_sync();
    const bool x_from_fwd = !XL1 && p.xt != nullptr;     // the forward kernel's bf16 X tile arrives by TMA with the delta tiles
    if constexpr (!XL1) {
    if (!x_from_fwd) load_norm_smem<N>(sNorm, p.nm, p.ns, p.D);
    for (int i = tid; i < (128 * 256 - (int)N::X_BYTES) / 16; i += 256) reinterpret_cast<uint4*>(sX + N::X_BYTES)[i] = make_uint4(0, 0, 0, 0);
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t TW2 = tmem, TW1 = tmem + 256;     // dW2^T halves [128 x U2] at +0, +128 ; dW1^T [128 x U1] at +256
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    float bsum1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    uint32_t phase = 0;
    bool first = true;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (!first) { mbar_wait(&bars[1], phase ^ 1); fence_after_sync(); }    // previous tile's MMAs done reading the tiles
        __syncthreads();
        TSTAMP();   // tile start (previous MMAs done)
        if (tid == 0) {
            mbar_expect_tx(&bars[0], N::A2_BYTES + 2 * N::A1_BYTES + (x_from_fwd ? N::X_BYTES : 0u));
            bulk_g2s(sD2, p.delta2 + (size_t)tile * N::A2_BYTES, N::A2_BYTES, &bars[0]);
            bulk_g2s(sD1, p.delta1 + (size_t)tile * N::A1_BYTES, N::A1_BYTES, &bars[0]);
            bulk_g2s(sA1, p.act1 + (size_t)tile * N::A1_BYTES, N::A1_BYTES, &bars[0]);
            if (x_from_fwd) bulk_g2s(sX, p.xt + (size_t)tile * N::X_BYTES, N::X_BYTES, &bars[0]);
        }
        if constexpr (!XL1) {
        if (!x_from_fwd) {
        const int m0 = tile * 128;
        stage_x_tile<N, 256>(sX, p.obs, chunk_row(m0, p.rows_per_chunk, p.chunk_stride), min(128, p.M - m0), p.D, sNorm, p.nm != nullptr);
        fence_async_smem();
        }
        }
        TSTAMP();   // X staged
        mbar_wait(&bars[0], phase);
        __syncthreads();
        TSTAMP();   // tile loads landed
        if (tid == 0) {
            fence_after_sync();
            const uint32_t acc = first ? 0u : 1u;
#pragma unroll
            for (int hh = 0; hh < N::U1 / 128; ++hh)
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    umma_bf16(TW2 + hh * N::U2, make_smem_desc(smem_u32(sA1) + hh * 16 * N::ACS + k * 256, 128, N::ACS),
                              make_smem_desc(smem_u32(sD2) + k * 256, 128, N::ACS), make_idesc_bf16(128, N::U2, 1, 1),
                              (acc || k > 0) ? 1u : 0u);
            if constexpr (!XL1) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                umma_bf16(TW1, make_smem_desc(smem_u32(sX) + k * 256, 128, N::ACS), make_smem_desc(smem_u32(sD1) + k * 256, 128, N::ACS),
                          make_idesc_bf16(128, N::U1, 1, 1), (acc || k > 0) ? 1u : 0u);
            }
            umma_commit(&bars[1]);
        }
        colsum8<128, N::U1 / 8, N::ACS, 256>(sD1, tid, bsum1);
        TSTAMP();   // bias sums done
        phase ^= 1;
        first = false;
    }
    float* part = p.part + (size_t)blockIdx.x * p.P;
    const bool native = p.u1 == N::U1 && p.u2 == N::U2;
    if (!first) {
        mbar_wait(&bars[1], phase ^ 1);
        fence_after_sync();
        TSTAMP();   // last MMAs done
        // dW2^T halves: lane = in index i (hh*128 + row), columns = out o: thread takes o in [64h, 64h+64)
#pragma unroll 1
        for (int hh = 0; hh < N::U1 / 128; ++hh) {
#pragma unroll 1
            for (int c0 = h * (N::U2 / 2); c0 < (h + 1) * (N::U2 / 2); c0 += 32) {
                float v[32];
                tmem_ld32(TW2 + hh * N::U2 + lane_base + c0, v);
                if (native) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) part[p.off_W2 + (size_t)(c0 + j) * N::U1 + hh * 128 + row] = v[j];
                } else if (hh * 128 + row < p.u1) {
                    float* dst = part + p.off_W2 + c0 * p.u1 + hh * 128 + row;
                    const int nv = p.u2 - c0;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < nv) dst[j * p.u1] = v[j];
                }
            }
        }
        // dW1^T: lane = in index i = row (< D valid), columns = out o in [128h, 128h+128)
        if constexpr (!XL1) {
#pragma unroll 1
        for (int c0 = h * (N::U1 / 2); c0 < (h + 1) * (N::U1 / 2); c0 += 32) {
            float v[32];
            tmem_ld32(TW1 + lane_base + c0, v);
            if (row < p.D) {
                float* dst = part + p.off_W1 + c0 * p.D + row;
                if (native) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) dst[j * p.D] = v[j];
                } else {
                    const int nv = p.u1 - c0;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < nv) dst[j * p.D] = v[j];
                }
            }
        }
        }
    } else {
        for (int i = tid; i < p.u2 * p.u1; i += 256) part[p.off_W2 + i] = 0.f;
        if (!XL1) for (int i = tid; i < p.u1 * p.D; i += 256) part[p.off_W1 + i] = 0.f;
    }
    {
        const int g = colsum8_owner_group<N::U1 / 8, 256>(tid);
        if (g >= 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (g * 8 + j < p.u1) part[p.off_b1 + g * 8 + j] = bsum1[j];
        }
    }
    fence_before_sync();
    __syncthreads();
    TSTAMP();   // flush done
    TSTAMP_END();
}

// ---- the whole backward pass in ONE launch: phase 1 = delta chain + dW3/dWh (bwd1_body), phase 2 = dW2/dW1 (bwd2_body).
//      Phase 2 of a CTA consumes only delta tiles that the SAME CTA produced in phase 1 (both phases walk the tiles
//      blockIdx.x, blockIdx.x + gridDim.x, ...), so no grid-wide synchronisation is needed -- only the generic-proxy stores
//      of delta1/delta2 must be ordered before the async-proxy (TMA) loads that read them back.
struct BwdArgs { Bwd1Args a; Bwd2Args b; };

template <class N, bool XL1 = false>
__global__ void __launch_bounds__(256, 1) mlp_bwd_tc_kernel(const BwdArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t tmem_slot;
    const uint32_t tmem = bwd_tmem_alloc(&tmem_slot);
    bwd1_body<N>(p.a, smem, tmem);
    __threadfence();
    asm volatile("fence.proxy.async.global;" ::: "memory");
    fence_async_smem();          // phase 2 re-uses the shared memory of phase 1 as TMA destinations
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    bwd2_body<N, XL1>(p.b, smem, tmem);
    if ((threadIdx.x >> 5) == 0) tmem_dealloc(tmem, 512);
}

// ---- backward 2, pipelined edition: the row index is the GEMM K dimension here, so the 128-row tiles are consumed as 64-row
//      half tiles through a two-stage TMA ring (96 KB per stage): the loads of half j+1 / j+2 are in flight while half j is
//      multiplied.  The normalised bf16 observation tile comes from the forward kernel (p.xt) instead of being re-derived.
struct Bwd2DbArgs {
    const uint8_t* xt; const uint8_t* act1; const uint8_t* delta2; const uint8_t* delta1; float* part;
    int M; int D; int P; int off_W2, off_W1, off_b1;
};

template <class N>
__global__ void __launch_bounds__(256, 1) mlp_bwd2_db_tc_kernel(const Bwd2DbArgs p) {
    constexpr uint32_t HCS = 1024;                                   // column-group stride of a 64-row half tile (64 rows x 16 B)
    constexpr uint32_t D2H = N::A2_BYTES / 2, D1H = N::A1_BYTES / 2, A1H = N::A1_BYTES / 2, XH = 16 * HCS;   // X half padded to 128 columns
    constexpr uint32_t STAGE = D2H + D1H + A1H + XH;
    constexpr int NCGX = N::DPAD / 8;                                // real column groups of the X tile
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * STAGE);  // [0,1] stage full, [2,3] stage consumed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    const int n_tiles = (p.M + 127) / 128;
    int n_stamp = 0; (void)n_stamp;
    constexpr int TSB = 256; (void)TSB;
    TSTAMP();   // kernel start
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
        fence_mbar_init();
    }
    // zero the padding column groups of both X half tiles once (the TMA copies only ever write the real ones)
    for (int s = 0; s < 2; ++s) {
        uint8_t* sX = smem + s * STAGE + D2H + D1H + A1H;
        for (int i = tid; i < (int)(XH - NCGX * HCS) / 16; i += 256) reinterpret_cast<uint4*>(sX + NCGX * HCS)[i] = make_uint4(0, 0, 0, 0);
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    pdl_sync();      // CTA-local set-up above; the delta tiles below are the predecessor's output
    const uint32_t tmem = *tmem_slot;
    const uint32_t TW2 = tmem, TW1 = tmem + 256;     // dW2^T halves [128 x U2] at +0, +128 ; dW1^T [128 x U1] at +256
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const int nt = ((int)blockIdx.x < n_tiles) ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int nh = 2 * nt;                            // half tiles of this CTA
    // warp 0 issues the copies of half tile j into stage j & 1: one 1 KB bulk copy per column group
    auto issue = [&](int j) {
        const int s = j & 1, hf = j & 1;
        const size_t tile = (size_t)blockIdx.x + (size_t)(j >> 1) * gridDim.x;
        uint8_t* sD2 = smem + s * STAGE; uint8_t* sD1 = sD2 + D2H; uint8_t* sA1 = sD1 + D1H; uint8_t* sX = sA1 + A1H;
        if (lane == 0) mbar_expect_tx(&bars[s], D2H + D1H + A1H + NCGX * HCS);
        __syncwarp();
        const uint8_t* gD2 = p.delta2 + tile * N::A2_BYTES + hf * HCS;
        const uint8_t* gD1 = p.delta1 + tile * N::A1_BYTES + hf * HCS;
        const uint8_t* gA1 = p.act1 + tile * N::A1_BYTES + hf * HCS;
        const uint8_t* gX = p.xt + tile * N::X_BYTES + hf * HCS;
        for (int g = lane; g < N::U1 / 8; g += 32) {
            bulk_g2s(sD1 + g * HCS, gD1 + (size_t)g * N::ACS, HCS, &bars[s]);
            bulk_g2s(sA1 + g * HCS, gA1 + (size_t)g * N::ACS, HCS, &bars[s]);
        }
        for (int g = lane; g < N::U2 / 8; g += 32) bulk_g2s(sD2 + g * HCS, gD2 + (size_t)g * N::ACS, HCS, &bars[s]);
        for (int g = lane; g < NCGX; g += 32) bulk_g2s(sX + g * HCS, gX + (size_t)g * N::ACS, HCS, &bars[s]);
    };
    if (warp == 0) {
        if (nh > 0) issue(0);
        if (nh > 1) issue(1);
    }
    float bsum1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    uint32_t ph_full = 0, ph_done = 0;     // bit s = phase parity of stage s's barrier
    for (int j = 0; j < nh; ++j) {
        const int s = j & 1;
        uint8_t* sD2 = smem + s * STAGE; uint8_t* sD1 = sD2 + D2H; uint8_t* sA1 = sD1 + D1H; uint8_t* sX = sA1 + A1H;
        TSTAMP();   // half start
        mbar_wait(&bars[s], (ph_full >> s) & 1u);
        ph_full ^= 1u << s;
        TSTAMP();   // loads landed
        if (tid == 0) {
            fence_after_sync();
            const uint32_t acc = j > 0 ? 1u : 0u;
#pragma unroll
            for (int hh = 0; hh < N::U1 / 128; ++hh)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    umma_bf16(TW2 + hh * N::U2, make_smem_desc(smem_u32(sA1) + hh * 16 * HCS + k * 256, 128, HCS),
                              make_smem_desc(smem_u32(sD2) + k * 256, 128, HCS), make_idesc_bf16(128, N::U2, 1, 1), (acc || k > 0) ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                umma_bf16(TW1, make_smem_desc(smem_u32(sX) + k * 256, 128, HCS), make_smem_desc(smem_u32(sD1) + k * 256, 128, HCS),
                          make_idesc_bf16(128, N::U1, 1, 1), (acc || k > 0) ? 1u : 0u);
            umma_commit(&bars[2 + s]);
        }
        colsum8<64, N::U1 / 8, HCS, 256>(sD1, tid, bsum1);     // bias gradient of layer 1: column sums of the d1 half tile
        if (j + 2 < nh) {
            // refill this stage with half j + 2 once its MMAs have consumed it and every thread is done with the column sums
            mbar_wait(&bars[2 + s], (ph_done >> s) & 1u);
            ph_done ^= 1u << s;
            fence_async_smem();
            __syncthreads();
            if (warp == 0) issue(j + 2);
        }
        TSTAMP();   // half done
    }
    float* part = p.part + (size_t)blockIdx.x * p.P;
    if (nh > 0) {
        // the last commit covers every earlier MMA
        const int sl = (nh - 1) & 1;
        mbar_wait(&bars[2 + sl], (ph_done >> sl) & 1u);
        if (nh > 1) mbar_wait(&bars[2 + (sl ^ 1)], (ph_done >> (sl ^ 1)) & 1u);
        fence_after_sync();
        TSTAMP();   // last MMAs done
#pragma unroll 1
        for (int hh = 0; hh < N::U1 / 128; ++hh) {
#pragma unroll 1
            for (int c0 = h * (N::U2 / 2); c0 < (h + 1) * (N::U2 / 2); c0 += 32) {
                float v[32];
                tmem_ld32(TW2 + hh * N::U2 + lane_base + c0, v);
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) part[p.off_W2 + (size_t)(c0 + jj) * N::U1 + hh * 128 + row] = v[jj];
            }
        }
#pragma unroll 1
        for (int c0 = h * (N::U1 / 2); c0 < (h + 1) * (N::U1 / 2); c0 += 32) {
            float v[32];
            tmem_ld32(TW1 + lane_base + c0, v);
            if (row < p.D) {
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) part[p.off_W1 + (size_t)(c0 + jj) * p.D + row] = v[jj];
            }
        }
    } else {
        for (int i = tid; i < N::U2 * N::U1; i += 256) part[p.off_W2 + i] = 0.f;
        for (int i = tid; i < N::U1 * p.D; i += 256) part[p.off_W1 + i] = 0.f;
    }
    {
        const int g = colsum8_owner_group<N::U1 / 8, 256>(tid);
        if (g >= 0) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) part[p.off_b1 + g * 8 + jj] = bsum1[jj];
        }
    }
    fence_before_sync();
    __syncthreads();
    TSTAMP();   // flush done
    TSTAMP_END();
    if (warp == 0) tmem_dealloc(tmem, 512);
}


// ================================================================================================= wide observations: layer 1
// a1 = elu(norm(obs) . W1^T + b1) for 64 < D <= 256 as a kernel of its own: W1 (U1 x DPAD bf16, 128 KB) stays resident, the whole
// normalised bf16 X tile (128 x DPAD, 64 KB) is staged per tile, one K = DPAD chain of MMAs fills T1[128, U1], and the epilogue
// writes the bf16 a1 tile straight to the global tiled buffer the chain kernels read (act1 during training, a scratch during the
// rollout).  Same operand layouts, descriptors and epilogue as layer 1 of mlp_fwd_tc_kernel.
struct L1FwdArgs {
    const float* obs; int rows_per_chunk; int64_t chunk_stride; int D; const float* nm; const float* ns;
    const uint8_t* wpack; const float* b1; int M; uint8_t* act1; int u1, act;
    uint8_t* xt;      // optional: normalised bf16 observation tiles (128 x DPAD) for l1_wgrad_tc_kernel
};

template <class N>
__global__ void __launch_bounds__(FWD_THREADS, 1) l1_fwd_tc_kernel(const L1FwdArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sW1 = smem; uint8_t* sX = sW1 + N::W1_BYTES;
    float* sB1 = reinterpret_cast<float*>(sX + N::X_BYTES);
    float* sNorm = sB1 + N::U1;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sNorm + 2 * N::DPAD);       // [0] W1, [1] mma
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    const int n_tiles = (p.M + 127) / 128;
    if (warp == 0) tmem_alloc(tmem_slot, 256);
    if (tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    pdl_sync();
    if (tid == 0) {
        mbar_expect_tx(&bars[0], N::W1_BYTES);
        bulk_g2s(sW1, p.wpack + N::W1_OFF, N::W1_BYTES, &bars[0]);
    }
    for (int i = tid; i < N::U1; i += FWD_THREADS) sB1[i] = i < p.u1 ? __ldg(p.b1 + i) : 0.f;
    load_norm_smem<N>(sNorm, p.nm, p.ns, p.D);
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t T1 = *tmem_slot;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t phase = 0;
    bool weights_ready = false;
    constexpr int NCGP = 16;       // column groups per staging pass: 128 columns, 4 x 32 B in flight per thread
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int m0 = tile * 128;
        const int rows_valid = min(128, p.M - m0);
        const int64_t arow0 = chunk_row(m0, p.rows_per_chunk, p.chunk_stride);
#pragma unroll 1
        for (int cg = 0; cg < N::DPAD / 8; cg += NCGP)
            stage_x_cols<N, FWD_THREADS, NCGP>(sX, p.obs, arow0, rows_valid, p.D, sNorm, p.nm != nullptr, cg, tid);
        fence_async_smem();
        if (!weights_ready) { mbar_wait(&bars[0], 0); weights_ready = true; }
        __syncthreads();
        if (tid == 0) {
            if (p.xt) {      // keep the normalised bf16 tile for the weight-gradient kernel: one 64 KB bulk store, asynchronous
                bulk_s2g(p.xt + (size_t)tile * N::X_BYTES, sX, N::X_BYTES);
                bulk_commit();
            }
            fence_after_sync();
            constexpr uint32_t idesc = make_idesc_bf16(128, N::U1, 0, 0);
#pragma unroll
            for (int k = 0; k < N::DPAD / 16; ++k)
                umma_bf16(T1, make_smem_desc(smem_u32(sX) + k * 2 * N::ACS, N::ACS, N::ARS),
                          make_smem_desc(smem_u32(sW1) + k * 2 * N::W1_CS, N::W1_CS, 128), idesc, k > 0);
            umma_commit(&bars[1]);
        }
        mbar_wait(&bars[1], phase);
        fence_after_sync();
        {
            uint8_t* g1 = p.act1 + (size_t)tile * N::A1_BYTES;
#pragma unroll 1
            for (int c0 = h * (N::U1 / 4); c0 < (h + 1) * (N::U1 / 4); c0 += 32) {
                float v[32];
                tmem_ld32(T1 + lane_base + c0, v);
                bias_act<32>(v, sB1 + c0);
                store_chunks32(v, row, c0, nullptr, g1);
            }
        }
        if (p.xt && tid == 0) bulk_wait_read0();      // the tile's copy-out (issued before the MMAs) has finished reading sX
        fence_before_sync();
        __syncthreads();       // T1 and the X tile are free for the next tile
        fence_after_sync();
        phase ^= 1;
    }
    if (!weights_ready) mbar_wait(&bars[0], 0);
    if (p.xt && tid == 0) bulk_wait_read0();          // shared memory must outlive the last copy-out's reads
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(T1, 256);
}

// dW1^T[i][o] = sum_r x[r][i] d1[r][o] for wide observations: DPAD / 128 halves of the `in` index, each a [128 x U1] fp32
// accumulator (2 x 256 = all 512 TMEM columns at DPAD = 256).  The delta-1 tiles come from the backward chain kernel (global,
// TMA), the X tile is re-derived from the observations.  Same MN-major operand trick and coalesced flush as bwd2_body.
struct L1WgradArgs {
    const float* obs; int rows_per_chunk; int64_t chunk_stride; int D; const float* nm; const float* ns;
    const uint8_t* delta1; float* part; int M; int P; int off_W1; int u1;
    const uint8_t* xt;      // optional: the tiles l1_fwd_tc_kernel emitted (TMA-loaded instead of re-deriving X from the fp32 observations)
};

template <class N>
__global__ void __launch_bounds__(256, 1) l1_wgrad_tc_kernel(const L1WgradArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t tmem_slot;
    constexpr int NH = N::DPAD / 128;
    static_assert(N::DPAD % 128 == 0 && NH * N::U1 <= 512, "dW1^T halves must fit the 512 TMEM columns");
    uint8_t* sD1 = smem; uint8_t* sX = sD1 + N::A1_BYTES;
    float* sNorm = reinterpret_cast<float*>(sX + N::X_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sNorm + 2 * N::DPAD);       // [0] tile load, [1] mma
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    const int n_tiles = (p.M + 127) / 128;
    const uint32_t tmem = bwd_tmem_alloc(&tmem_slot);
    if (tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    pdl_sync();
    load_norm_smem<N>(sNorm, p.nm, p.ns, p.D);
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t phase = 0;
    bool first = true;
    constexpr int NCGP = 16;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (!first) { mbar_wait(&bars[1], phase ^ 1); fence_after_sync(); }    // previous tile's MMAs done reading the tiles
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&bars[0], N::A1_BYTES + (p.xt ? N::X_BYTES : 0u));
            bulk_g2s(sD1, p.delta1 + (size_t)tile * N::A1_BYTES, N::A1_BYTES, &bars[0]);
            if (p.xt) bulk_g2s(sX, p.xt + (size_t)tile * N::X_BYTES, N::X_BYTES, &bars[0]);
        }
        if (!p.xt) {
        const int m0 = tile * 128;
#pragma unroll 1
        for (int cg = 0; cg < N::DPAD / 8; cg += NCGP)
            stage_x_cols<N, 256, NCGP>(sX, p.obs, chunk_row(m0, p.rows_per_chunk, p.chunk_stride), min(128, p.M - m0), p.D, sNorm,
                                       p.nm != nullptr, cg, tid);
        fence_async_smem();
        }
        mbar_wait(&bars[0], phase);
        __syncthreads();
        if (tid == 0) {
            fence_after_sync();
            const uint32_t acc = first ? 0u : 1u;
#pragma unroll
            for (int hh = 0; hh < NH; ++hh)
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    umma_bf16(tmem + hh * N::U1, make_smem_desc(smem_u32(sX) + hh * 16 * N::ACS + k * 256, 128, N::ACS),
                              make_smem_desc(smem_u32(sD1) + k * 256, 128, N::ACS), make_idesc_bf16(128, N::U1, 1, 1),
                              (acc || k > 0) ? 1u : 0u);
            umma_commit(&bars[1]);
        }
        phase ^= 1;
        first = false;
    }
    float* part = p.part + (size_t)blockIdx.x * p.P;
    if (!first) {
        mbar_wait(&bars[1], phase ^ 1);
        fence_after_sync();
        // lane = in index i = hh * 128 + row (< D valid), columns = out o: thread takes o in [128h, 128h + 128)
#pragma unroll 1
        for (int hh = 0; hh < NH; ++hh) {
            const int i = hh * 128 + row;
#pragma unroll 1
            for (int c0 = h * (N::U1 / 2); c0 < (h + 1) * (N::U1 / 2); c0 += 32) {
                float v[32];
                tmem_ld32(tmem + hh * N::U1 + lane_base + c0, v);
                if (i < p.D) {
                    float* dst = part + p.off_W1 + c0 * p.D + i;
                    const int nv = p.u1 - c0;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < nv) dst[j * p.D] = v[j];
                }
            }
        }
    } else {
        for (int i = tid; i < p.u1 * p.D; i += 256) part[p.off_W1 + i] = 0.f;
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

template <class N, bool XL1 = false> constexpr size_t fwd_smem() {
    return (XL1 ? (size_t)N::W2_BYTES + N::W3_BYTES + N::WH_BYTES + N::A1_BYTES + N::A2_BYTES + N::A3_BYTES
                : (size_t)N::PACK_BYTES + N::A1_BYTES + (N::A2_BYTES > N::X_BYTES ? N::A2_BYTES : N::X_BYTES)) +
           sizeof(float) * (N::U1 + N::U2 + N::U3 + N::AP + 64 + 2 * N::DPAD + 4 * LOSS_SLOTS) + sizeof(double) * LOSS_SLOTS + 8 * 8 + 16;
}
template <class N> constexpr size_t l1_fwd_smem() { return (size_t)N::W1_BYTES + N::X_BYTES + sizeof(float) * (N::U1 + 2 * N::DPAD) + 2 * 8 + 16; }
template <class N> constexpr size_t l1_wgrad_smem() { return (size_t)N::A1_BYTES + N::X_BYTES + sizeof(float) * 2 * N::DPAD + 2 * 8 + 16; }
template <class N> constexpr size_t bwd1_smem() {
    return (size_t)N::WH_BYTES + N::W3_BYTES + N::W2_BYTES + N::DH_BYTES + 128 * 256 + N::A2_BYTES + N::A3_BYTES + N::A2_BYTES + 8 * 8 + 16;
}
template <class N> constexpr size_t bwd2_db_smem() { return (size_t)2 * (N::A2_BYTES / 2 + N::A1_BYTES + 16 * 1024) + 4 * 8 + 16; }
template <class N, bool XL1 = false> constexpr size_t bwd2_smem() {
    return (size_t)N::A2_BYTES + 2 * N::A1_BYTES + (XL1 ? 0 : 128 * 256 + sizeof(float) * 2 * N::DPAD) + 4 * 8 + 16;
}
template <class N, bool XL1 = false> constexpr size_t bwd_smem() {
    return bwd1_smem<N>() > bwd2_smem<N, XL1>() ? bwd1_smem<N>() : bwd2_smem<N, XL1>();
}

// Persistent grid for n_tiles row tiles on 148 SMs: the number of waves w = ceil(n_tiles / 148) fixes the critical path; the FEWEST
// CTAs with that many waves (ceil(n_tiles / w)) give every CTA the same tile count and -- for the backward kernels -- the fewest
// split-gradient rows for the reducer to read (c2 minibatch: 256 tiles -> 128 CTAs x 2 tiles instead of 148 rows).
static inline int tc_grid(int n_tiles) {
    const int waves = (n_tiles + 147) / 148;
    return (n_tiles + waves - 1) / waves;
}

// Geometries: any three-layer MLP that fits the compiled tile widths (u1 <= 256, u2 <= 128, u3 <= 64, up to 15 actions) runs on the
// kernels compiled for [256, 128, 64]: the packed bf16 weights are zero-padded to the tile widths (pack_weights_kernel), padded units
// have zero weights and zero bias, so their activations (elu / relu / tanh of 0) and their deltas are exactly zero, and every flush
// writes with the LOGICAL strides of the fp32 parameter arena.  [128, 64, 32] (e.g. configs/mujoco/walker2d.yaml) runs this way.
bool net_fits(int u1, int u2, int u3, int A) { return u1 >= 1 && u2 >= 1 && u3 >= 1 && u1 <= 256 && u2 <= 128 && u3 <= 64 && A >= 1 && A + 1 <= 16; }
bool net_is_native(int u1, int u2, int u3) { return u1 == 256 && u2 == 128 && u3 == 64; }
bool net_is_c2(int D, int u1, int u2, int u3, int A) { return D >= 1 && D <= 64 && net_fits(u1, u2, u3, A); }
// wide observations: the same hidden layers, layer 1 in its own kernels (NetW)
bool net_is_wide(int D, int u1, int u2, int u3, int A) { return D > 64 && D <= 256 && net_fits(u1, u2, u3, A); }
int net_kind(int D, int u1, int u2, int u3, int A) { return net_is_c2(D, u1, u2, u3, A) ? 1 : (net_is_wide(D, u1, u2, u3, A) ? 2 : 0); }

template <class N>
void fill_pack_table(int D, int u1, int u2, int u3, int A, int off_W1, int off_W2, int off_W3, int off_Wh, b200rl_pack_table* out_host) {
    out_host->n_seg = 4;
    const int offs[4] = {off_W1, off_W2, off_W3, off_Wh};
    const int rows[4] = {u1, u2, u3, A + 1}, cols[4] = {D, u1, u2, u3};
    const unsigned cs[4] = {N::W1_CS, N::W2_CS, N::W3_CS, N::WH_CS}, dst[4] = {N::W1_OFF, N::W2_OFF, N::W3_OFF, N::WH_OFF};
    for (int i = 0; i < 4; ++i) {
        out_host->flat_off[i] = offs[i]; out_host->rows[i] = rows[i]; out_host->cols[i] = cols[i];
        out_host->cs_bytes[i] = cs[i]; out_host->dst_off[i] = dst[i];
    }
}

template <class N>
int pack_weights_impl(const float* W1, const float* W2, const float* W3, const float* W_head, int D, int u1, int u2, int u3, int A,
                      void* wpack, void* stream) {
    PackArgs a;
    a.seg[0] = PackSeg{W1, u1, D, N::U1, N::DPAD, N::W1_OFF};
    a.seg[1] = PackSeg{W2, u2, u1, N::U2, N::U1, N::W2_OFF};
    a.seg[2] = PackSeg{W3, u3, u2, N::U3, N::U2, N::W3_OFF};
    a.seg[3] = PackSeg{W_head, A + 1, u3, N::AP, N::U3, N::WH_OFF};
    pack_weights_kernel<<<dim3(16, 4), 256, 0, as_stream(stream)>>>(a, (uint8_t*)wpack);
    B200RL_LAUNCH_CHECK();
    return B200RL_OK;
}

// layer 1 of the wide path (see l1_fwd_tc_kernel): a1 tiles of M rows into `act1`
template <class N>
int launch_l1_fwd(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D, const float* nm, const float* ns, const void* wpack,
                  const float* b1, int M, void* act1, int u1, int act, void* xt, void* stream) {
    const int n_tiles = (M + 127) / 128;
    const int grid = tc_grid(n_tiles);
    L1FwdArgs a{obs, rows_per_chunk, chunk_stride, D, nm, ns, (const uint8_t*)wpack, b1, M, (uint8_t*)act1, u1, act, (uint8_t*)xt};
    constexpr size_t smem = l1_fwd_smem<N>();
    static_assert(smem <= 227 * 1024, "layer-1 forward kernel shared memory budget");
    cudaError_t e = cudaFuncSetAttribute(l1_fwd_tc_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = launch_k(l1_fwd_tc_kernel<N>, dim3(grid), dim3(FWD_THREADS), smem, as_stream(stream), a);
    return e == cudaSuccess ? B200RL_OK : (int)e;
}

}  // namespace

// ------------------------------------------------------------------------------------------------- C ABI
#ifdef B200RL_TC_MAIN
// 0 = no tcgen05 kernels for this geometry; 1 = resident-weights kernels (obs <= 64); 2 = wide observations (64 < obs <= 256):
// layer 1 in its own kernels
B200RL_EXPORT int b200rl_tc_supported(int D, int u1, int u2, int u3, int A) { return net_kind(D, u1, u2, u3, A); }

B200RL_EXPORT int64_t b200rl_tc_pack_bytes(int D, int u1, int u2, int u3, int A) {
    const int kind = net_kind(D, u1, u2, u3, A);
    return kind == 1 ? (int64_t)NetC2::PACK_BYTES : (kind == 2 ? (int64_t)NetW::PACK_BYTES : -1);
}
// bytes of one 128-row tile of: act1, act2, act3, d_head  (tiled INTERLEAVE bf16 buffers)
B200RL_EXPORT int b200rl_tc_tile_bytes(int D, int u1, int u2, int u3, int A, int64_t* out4_host) {
    if (!net_kind(D, u1, u2, u3, A) || !out4_host) return B200RL_EUNSUPPORTED;       // the activation tiles do not depend on DPAD
    out4_host[0] = NetC2::A1_BYTES; out4_host[1] = NetC2::A2_BYTES; out4_host[2] = NetC2::A3_BYTES; out4_host[3] = NetC2::DH_BYTES;
    return B200RL_OK;
}

B200RL_EXPORT int64_t b200rl_tc_xtile_bytes(int D, int u1, int u2, int u3, int A) {
    const int kind = net_kind(D, u1, u2, u3, A);
    return kind == 1 ? (int64_t)NetC2::X_BYTES : (kind == 2 ? (int64_t)NetW::X_BYTES : -1);
}

// segments of the packed weight buffer, for the optimiser's fused refresh (b200rl_adam_step_f32)
B200RL_EXPORT int b200rl_tc_pack_table(int D, int u1, int u2, int u3, int A, int off_W1, int off_W2, int off_W3, int off_Wh,
                                       b200rl_pack_table* out_host) {
    if (!out_host) return B200RL_EINVAL;
    const int kind = net_kind(D, u1, u2, u3, A);
    if (!kind) return B200RL_EUNSUPPORTED;
    if (kind == 1) fill_pack_table<NetC2>(D, u1, u2, u3, A, off_W1, off_W2, off_W3, off_Wh, out_host);
    else fill_pack_table<NetW>(D, u1, u2, u3, A, off_W1, off_W2, off_W3, off_Wh, out_host);
    return B200RL_OK;
}

B200RL_EXPORT int b200rl_tc_pack_weights(const float* W1, const float* W2, const float* W3, const float* W_head,
                                         int D, int u1, int u2, int u3, int A, void* wpack, void* stream) {
    if (!W1 || !W2 || !W3 || !W_head || !wpack) return B200RL_EINVAL;
    const int kind = net_kind(D, u1, u2, u3, A);
    if (!kind) return B200RL_EUNSUPPORTED;
    return kind == 1 ? pack_weights_impl<NetC2>(W1, W2, W3, W_head, D, u1, u2, u3, A, wpack, stream)
                     : pack_weights_impl<NetW>(W1, W2, W3, W_head, D, u1, u2, u3, A, wpack, stream);
}

#endif  // B200RL_TC_MAIN

static int tc_check_rows(int M, int rows_per_chunk) {
    if (M <= 0 || rows_per_chunk <= 0) return B200RL_EINVAL;
    if (M > rows_per_chunk && rows_per_chunk % 128 != 0) return B200RL_EUNSUPPORTED;   // tiles may not straddle chunks
    return B200RL_OK;
}

extern "C" int TCIMPL(b200rl_tcimpl_fwd_train)(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D,
                                          const float* norm_mean, const float* norm_std, const void* wpack,
                                          const float* b1, const float* b2, const float* b3, const float* b_head, const float* logstd,
                                          int u1, int u2, int u3, int activation, int M, int A,
                                          const float* actions, float* old_mu, float* old_sigma, const float* old_values_n,
                                          const float* returns_n, const float* old_neglogp, const float* advs_n, const float* mask,
                                          const b200rl_loss_cfg* cfg_host, const float* inv_count_dev,
                                          void* act1, void* act2, void* act3, void* dhead, void* xtile,
                                          double* partials, int max_partials, int* n_blocks_out_host, void* stream) {
    if (!obs || !wpack || !b1 || !b2 || !b3 || !b_head || !logstd || !actions || !old_mu || !old_sigma || !old_values_n || !returns_n ||
        !old_neglogp || !advs_n || !cfg_host || !act1 || !act2 || !act3 || !dhead || !partials)
        return B200RL_EINVAL;
    const int kind = net_kind(D, u1, u2, u3, A);
    if (!kind || activation != TC_ACT) return B200RL_EUNSUPPORTED;
    int rc = tc_check_rows(M, rows_per_chunk);
    if (rc) return rc;
    const int n_tiles = (M + 127) / 128;
    const int grid = tc_grid(n_tiles);
    if (n_blocks_out_host) *n_blocks_out_host = grid;
    if (grid > max_partials) return B200RL_EINVAL;
    FwdArgs p{};
    p.obs = obs; p.rows_per_chunk = rows_per_chunk; p.chunk_stride = chunk_stride; p.D = D; p.nm = norm_mean; p.ns = norm_std;
    p.wpack = (const uint8_t*)wpack; p.b1 = b1; p.b2 = b2; p.b3 = b3; p.bh = b_head; p.logstd = logstd; p.M = M; p.A = A;
    p.u1 = u1; p.u2 = u2; p.u3 = u3; p.act = activation;
    p.la = LossArena{actions, old_mu, old_sigma, old_values_n, returns_n, old_neglogp, advs_n, mask};
    p.inv_count_dev = inv_count_dev;
    p.cfg = LossCfgDev{cfg_host->e_clip, cfg_host->critic_coef, cfg_host->bounds_loss_coef, cfg_host->has_bounds_loss,
                       cfg_host->bound_loss_type, cfg_host->clip_value, cfg_host->use_smooth_clamp, cfg_host->ppo,
                       log1pf(-cfg_host->e_clip), log1pf(cfg_host->e_clip)};
    p.act1 = (uint8_t*)act1; p.act2 = (uint8_t*)act2; p.act3 = (uint8_t*)act3; p.dhead = (uint8_t*)dhead; p.partials = partials;
    p.xt = (uint8_t*)xtile;
    if (kind == 2) {
        // wide observations: layer 1 (a1 tiles -> act1), then the chain kernel in its external-layer-1 form
        rc = launch_l1_fwd<NetW>(obs, rows_per_chunk, chunk_stride, D, norm_mean, norm_std, wpack, b1, M, act1, u1, activation, xtile, stream);
        if (rc) return rc;
        constexpr size_t smemw = fwd_smem<NetW, true>();
        static_assert(smemw <= 227 * 1024, "forward kernel (external layer 1) shared memory budget");
        cudaError_t ew = cudaFuncSetAttribute(mlp_fwd_tc_kernel<NetW, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw);
        if (ew != cudaSuccess) return (int)ew;
        ew = launch_k(mlp_fwd_tc_kernel<NetW, true, true>, dim3(grid), dim3(FWD_THREADS), smemw, as_stream(stream), p);
        return ew == cudaSuccess ? B200RL_OK : (int)ew;
    }
    using N = NetC2;
    constexpr size_t smem = fwd_smem<N>();
    static_assert(smem <= 227 * 1024, "forward kernel shared memory budget");
    cudaError_t e = cudaFuncSetAttribute(mlp_fwd_tc_kernel<N, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = launch_k(mlp_fwd_tc_kernel<N, true>, dim3(grid), dim3(FWD_THREADS), smem, as_stream(stream), p);
    if (e != cudaSuccess) return (int)e;
    return B200RL_OK;
}

extern "C" int TCIMPL(b200rl_tcimpl_fwd_rollout)(const float* obs, int D, const float* norm_mean, const float* norm_std, const void* wpack,
                                            const float* b1, const float* b2, const float* b3, const float* b_head, const float* logstd,
                                            int u1, int u2, int u3, int activation, int N_rows, int A,
                                            const double* vms_mean, const double* vms_var, int normalize_value,
                                            const float* noise, uint64_t seed, const uint64_t* rng_epoch_dev, uint32_t step_index,
                                            float* actions, float* mus, float* sigmas, float* neglogp, float* values,
                                            float* env_actions, int clip_actions, const float* act_low, const float* act_high,
                                            const uint8_t* dones_cur, uint8_t* dones_out, const float* prev_dones, float* valid_out,
                                            int values_only, void* l1_scratch, void* stream) {
    if (!obs || !wpack || !b1 || !b2 || !b3 || !b_head || !logstd || !values || N_rows <= 0) return B200RL_EINVAL;
    if (!values_only && (!actions || !mus || !sigmas || !neglogp)) return B200RL_EINVAL;
    if (normalize_value && (!vms_mean || !vms_var)) return B200RL_EINVAL;
    if (env_actions && clip_actions && (!act_low || !act_high)) return B200RL_EINVAL;
    if (dones_out && !dones_cur) return B200RL_EINVAL;
    const int kind = net_kind(D, u1, u2, u3, A);
    if (!kind || activation != TC_ACT) return B200RL_EUNSUPPORTED;
    if (kind == 2 && !l1_scratch) return B200RL_EINVAL;
    const int n_tiles = (N_rows + 127) / 128;
    const int grid = tc_grid(n_tiles);
    FwdArgs p{};
    p.obs = obs; p.rows_per_chunk = N_rows; p.chunk_stride = 0; p.D = D; p.nm = norm_mean; p.ns = norm_std;
    p.wpack = (const uint8_t*)wpack; p.b1 = b1; p.b2 = b2; p.b3 = b3; p.bh = b_head; p.logstd = logstd; p.M = N_rows; p.A = A;
    p.u1 = u1; p.u2 = u2; p.u3 = u3; p.act = activation;
    p.vms_mean = vms_mean; p.vms_var = vms_var; p.normalize_value = normalize_value; p.noise = noise; p.seed = seed;
    p.rng_epoch = rng_epoch_dev; p.step_index = step_index; p.actions = actions; p.mus = mus; p.sigmas = sigmas; p.neglogp = neglogp;
    p.values = values; p.env_actions = env_actions; p.clip_actions = clip_actions; p.act_low = act_low; p.act_high = act_high;
    p.dones_cur = dones_cur; p.dones_out = dones_out; p.prev_dones = prev_dones; p.valid_out = valid_out; p.values_only = values_only;
    if (kind == 2) {
        int rc = launch_l1_fwd<NetW>(obs, N_rows, 0, D, norm_mean, norm_std, wpack, b1, N_rows, l1_scratch, u1, activation, nullptr, stream);
        if (rc) return rc;
        p.act1 = (uint8_t*)l1_scratch;
        constexpr size_t smemw = fwd_smem<NetW, true>();
        cudaError_t ew = cudaFuncSetAttribute(mlp_fwd_tc_kernel<NetW, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw);
        if (ew != cudaSuccess) return (int)ew;
        ew = launch_k(mlp_fwd_tc_kernel<NetW, false, true>, dim3(grid), dim3(FWD_THREADS), smemw, as_stream(stream), p);
        return ew == cudaSuccess ? B200RL_OK : (int)ew;
    }
    using N = NetC2;
    constexpr size_t smem = fwd_smem<N>();
    cudaError_t e = cudaFuncSetAttribute(mlp_fwd_tc_kernel<N, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = launch_k(mlp_fwd_tc_kernel<N, false>, dim3(grid), dim3(FWD_THREADS), smem, as_stream(stream), p);
    if (e != cudaSuccess) return (int)e;
    return B200RL_OK;
}

extern "C" int TCIMPL(b200rl_tcimpl_bwd)(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D,
                                    const float* norm_mean, const float* norm_std, const void* wpack,
                                    int u1, int u2, int u3, int activation, int M, int A,
                                    const void* act1, const void* act2, const void* act3, const void* dhead, const void* xtile,
                                    int pipelined_wgrad, void* delta2, void* delta1, float* part, int max_parts, int P,
                                    int off_W1, int off_b1, int off_W2, int off_b2, int off_W3, int off_b3, int off_Wh, int off_bh,
                                    int* n_parts_out_host, void* stream) {
    if (!obs || !wpack || !act1 || !act2 || !act3 || !dhead || !delta2 || !delta1 || !part) return B200RL_EINVAL;
    const int kind = net_kind(D, u1, u2, u3, A);
    if (!kind || activation != TC_ACT) return B200RL_EUNSUPPORTED;
    if (pipelined_wgrad && (!xtile || kind == 2 || !net_is_native(u1, u2, u3))) return B200RL_EUNSUPPORTED;   // option of the native resident-W1 geometry, needs the X tiles
    int rc = tc_check_rows(M, rows_per_chunk);
    if (rc) return rc;
    using N = NetC2;
    const int n_tiles = (M + 127) / 128;
    const int grid = tc_grid(n_tiles);
    if (n_parts_out_host) *n_parts_out_host = grid;
    if (grid > max_parts) return B200RL_EINVAL;
    Bwd1Args a{(const uint8_t*)wpack, (const uint8_t*)act1, (const uint8_t*)act2, (const uint8_t*)act3, (const uint8_t*)dhead,
               (uint8_t*)delta2, (uint8_t*)delta1, part, M, A, P, off_W3, off_b3, off_b2, off_Wh, off_bh, u1, u2, u3, activation};
    cudaError_t e;
    if (pipelined_wgrad) {
        // two launches: delta chain, then the pipelined weight-gradient kernel (observation tiles from the forward kernel,
        // 64-row half tiles through a two-stage TMA ring)
        constexpr size_t smem1 = bwd1_smem<N>();
        static_assert(smem1 <= 227 * 1024, "bwd1 shared memory budget");
        e = cudaFuncSetAttribute(mlp_bwd1_tc_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
        if (e != cudaSuccess) return (int)e;
        e = launch_k(mlp_bwd1_tc_kernel<N>, dim3(grid), dim3(256), smem1, as_stream(stream), a);
        if (e != cudaSuccess) return (int)e;
        Bwd2DbArgs b{(const uint8_t*)xtile, (const uint8_t*)act1, (const uint8_t*)delta2, (const uint8_t*)delta1, part, M, D, P,
                     off_W2, off_W1, off_b1};
        constexpr size_t smem2 = bwd2_db_smem<N>();
        static_assert(smem2 <= 227 * 1024, "bwd2 (pipelined) shared memory budget");
        e = cudaFuncSetAttribute(mlp_bwd2_db_tc_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
        if (e != cudaSuccess) return (int)e;
        e = launch_k(mlp_bwd2_db_tc_kernel<N>, dim3(grid), dim3(256), smem2, as_stream(stream), b);
        if (e != cudaSuccess) return (int)e;
        return B200RL_OK;
    }
    if (kind == 2) {
        // wide observations: the chain kernel without the W1 part, then dW1 in its own kernel (same grid => same split rows)
        BwdArgs abw{a, Bwd2Args{obs, rows_per_chunk, chunk_stride, D, norm_mean, norm_std, (const uint8_t*)act1, (const uint8_t*)delta2,
                                (const uint8_t*)delta1, part, M, P, off_W2, off_W1, off_b1, u1, u2, nullptr}};
        constexpr size_t smemw = bwd_smem<NetW, true>();
        static_assert(smemw <= 227 * 1024, "backward kernel (external layer 1) shared memory budget");
        e = cudaFuncSetAttribute(mlp_bwd_tc_kernel<NetW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw);
        if (e != cudaSuccess) return (int)e;
        e = launch_k(mlp_bwd_tc_kernel<NetW, true>, dim3(grid), dim3(256), smemw, as_stream(stream), abw);
        if (e != cudaSuccess) return (int)e;
        L1WgradArgs w{obs, rows_per_chunk, chunk_stride, D, norm_mean, norm_std, (const uint8_t*)delta1, part, M, P, off_W1, u1, (const uint8_t*)xtile};
        constexpr size_t smem1w = l1_wgrad_smem<NetW>();
        static_assert(smem1w <= 227 * 1024, "layer-1 weight-gradient kernel shared memory budget");
        e = cudaFuncSetAttribute(l1_wgrad_tc_kernel<NetW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1w);
        if (e != cudaSuccess) return (int)e;
        e = launch_k(l1_wgrad_tc_kernel<NetW>, dim3(grid), dim3(256), smem1w, as_stream(stream), w);
        return e == cudaSuccess ? B200RL_OK : (int)e;
    }
    // default: the whole backward pass in one launch
    BwdArgs ab{a, Bwd2Args{obs, rows_per_chunk, chunk_stride, D, norm_mean, norm_std, (const uint8_t*)act1, (const uint8_t*)delta2,
                           (const uint8_t*)delta1, part, M, P, off_W2, off_W1, off_b1, u1, u2, (const uint8_t*)xtile}};
    constexpr size_t smem = bwd_smem<N>();
    static_assert(smem <= 227 * 1024, "backward kernel shared memory budget");
    e = cudaFuncSetAttribute(mlp_bwd_tc_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = launch_k(mlp_bwd_tc_kernel<N>, dim3(grid), dim3(256), smem, as_stream(stream), ab);
    if (e != cudaSuccess) return (int)e;
    return B200RL_OK;
}

#ifdef B200RL_TC_MAIN
// ---- dispatch on the MLP activation: one set of kernels per activation, compiled in its own translation unit ----
#define B200RL_TC_DECL(ACTN)                                                                                                                        \
    extern "C" int b200rl_tcimpl_fwd_train_act##ACTN(const float*, int, int64_t, int, const float*, const float*, const void*, const float*, const float*, \
                                                      const float*, const float*, const float*, int, int, int, int, int, int, const float*, float*, float*,  \
                                                      const float*, const float*, const float*, const float*, const float*, const b200rl_loss_cfg*,         \
                                                      const float*, void*, void*, void*, void*, void*, double*, int, int*, void*);                          \
    extern "C" int b200rl_tcimpl_fwd_rollout_act##ACTN(const float*, int, const float*, const float*, const void*, const float*, const float*, const float*, \
                                                        const float*, const float*, int, int, int, int, int, int, const double*, const double*, int,           \
                                                        const float*, uint64_t, const uint64_t*, uint32_t, float*, float*, float*, float*, float*, float*, int, \
                                                        const float*, const float*, const uint8_t*, uint8_t*, const float*, float*, int, void*, void*);         \
    extern "C" int b200rl_tcimpl_bwd_act##ACTN(const float*, int, int64_t, int, const float*, const float*, const void*, int, int, int, int, int, int,        \
                                                const void*, const void*, const void*, const void*, const void*, int, void*, void*, float*, int, int, int, int, \
                                                int, int, int, int, int, int, int*, void*);
B200RL_TC_DECL(1)
B200RL_TC_DECL(2)
B200RL_TC_DECL(3)
#undef B200RL_TC_DECL
#define B200RL_TC_DISPATCH(fn, ...)                                        \
    switch (activation) {                                                  \
        case B200RL_ACT_ELU: return fn##_act1(__VA_ARGS__);                \
        case B200RL_ACT_RELU: return fn##_act2(__VA_ARGS__);               \
        case B200RL_ACT_TANH: return fn##_act3(__VA_ARGS__);               \
        default: return B200RL_EUNSUPPORTED;                               \
    }

B200RL_EXPORT int b200rl_tc_mlp_fwd_train(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D,
                                          const float* norm_mean, const float* norm_std, const void* wpack,
                                          const float* b1, const float* b2, const float* b3, const float* b_head, const float* logstd,
                                          int u1, int u2, int u3, int activation, int M, int A,
                                          const float* actions, float* old_mu, float* old_sigma, const float* old_values_n,
                                          const float* returns_n, const float* old_neglogp, const float* advs_n, const float* mask,
                                          const b200rl_loss_cfg* cfg_host, const float* inv_count_dev,
                                          void* act1, void* act2, void* act3, void* dhead, void* xtile,
                                          double* partials, int max_partials, int* n_blocks_out_host, void* stream) {
    B200RL_TC_DISPATCH(b200rl_tcimpl_fwd_train, obs, rows_per_chunk, chunk_stride, D, norm_mean, norm_std, wpack, b1, b2, b3, b_head, logstd, u1, u2, u3,
                       activation, M, A, actions, old_mu, old_sigma, old_values_n, returns_n, old_neglogp, advs_n, mask, cfg_host, inv_count_dev, act1,
                       act2, act3, dhead, xtile, partials, max_partials, n_blocks_out_host, stream)
}

B200RL_EXPORT int b200rl_tc_mlp_fwd_rollout(const float* obs, int D, const float* norm_mean, const float* norm_std, const void* wpack,
                                            const float* b1, const float* b2, const float* b3, const float* b_head, const float* logstd,
                                            int u1, int u2, int u3, int activation, int N_rows, int A,
                                            const double* vms_mean, const double* vms_var, int normalize_value,
                                            const float* noise, uint64_t seed, const uint64_t* rng_epoch_dev, uint32_t step_index,
                                            float* actions, float* mus, float* sigmas, float* neglogp, float* values,
                                            float* env_actions, int clip_actions, const float* act_low, const float* act_high,
                                            const uint8_t* dones_cur, uint8_t* dones_out, const float* prev_dones, float* valid_out,
                                            int values_only, void* l1_scratch, void* stream) {
    B200RL_TC_DISPATCH(b200rl_tcimpl_fwd_rollout, obs, D, norm_mean, norm_std, wpack, b1, b2, b3, b_head, logstd, u1, u2, u3, activation, N_rows, A, vms_mean,
                       vms_var, normalize_value, noise, seed, rng_epoch_dev, step_index, actions, mus, sigmas, neglogp, values, env_actions, clip_actions,
                       act_low, act_high, dones_cur, dones_out, prev_dones, valid_out, values_only, l1_scratch, stream)
}

B200RL_EXPORT int b200rl_tc_mlp_bwd(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D,
                                    const float* norm_mean, const float* norm_std, const void* wpack,
                                    int u1, int u2, int u3, int activation, int M, int A,
                                    const void* act1, const void* act2, const void* act3, const void* dhead, const void* xtile,
                                    int pipelined_wgrad, void* delta2, void* delta1, float* part, int max_parts, int P,
                                    int off_W1, int off_b1, int off_W2, int off_b2, int off_W3, int off_b3, int off_Wh, int off_bh,
                                    int* n_parts_out_host, void* stream) {
    B200RL_TC_DISPATCH(b200rl_tcimpl_bwd, obs, rows_per_chunk, chunk_stride, D, norm_mean, norm_std, wpack, u1, u2, u3, activation, M, A, act1, act2, act3,
                       dhead, xtile, pipelined_wgrad, delta2, delta1, part, max_parts, P, off_W1, off_b1, off_W2, off_b2, off_W3, off_b3, off_Wh, off_bh,
                       n_parts_out_host, stream)
}
#undef B200RL_TC_DISPATCH

#ifdef B200RL_TEST_HOOKS   // test-only host entry points: compiled into tests/libb200rl_testhooks.so (csrc/build.py), not into the product library
// host test entry point (tests/test_tc_rows_cpu.py): the X-tile staging of the wide-observation kernels (stage_x_cols, __host__ __device__)
// run thread by thread on the CPU -- out_tile receives the 128 x 256 bf16 INTERLEAVE tile (64 KB).  n_threads: 512 (l1_fwd) or 256 (l1_wgrad).
B200RL_EXPORT int b200rl_hosttest_stage_x_cols(const float* obs, int64_t row0, int rows_valid, int D, const float* norm_mean, const float* norm_std,
                                               int n_threads, void* out_tile) {
    using N = NetW;
    if (!obs || !out_tile || D <= 0 || D > N::DPAD || (n_threads != 512 && n_threads != 256)) return B200RL_EINVAL;
    static float sNorm[2 * N::DPAD];
    for (int c = 0; c < N::DPAD; ++c) {          // load_norm_smem
        sNorm[c] = (norm_mean && c < D) ? norm_mean[c] : 0.f;
        sNorm[N::DPAD + c] = (norm_std && c < D) ? 1.0f / norm_std[c] : 1.f;
    }
    for (int cg = 0; cg < N::DPAD / 8; cg += 16)
        for (int tid = 0; tid < n_threads; ++tid) {
            if (n_threads == 512) stage_x_cols<N, 512, 16>((uint8_t*)out_tile, obs, row0, rows_valid, D, sNorm, norm_mean != nullptr, cg, tid);
            else stage_x_cols<N, 256, 16>((uint8_t*)out_tile, obs, row0, rows_valid, D, sNorm, norm_mean != nullptr, cg, tid);
        }
    return B200RL_OK;
}

// host test entry point (tests/test_tc_rows_cpu.py): the packed-weight layout of the wide net (NetW) produced by the SAME element rule as
// pack_weights_kernel (chunk (r, cg) of a [Rpad x Cpad] tile at cg * (Rpad / 8) * 128 + tile_off), on the CPU.
B200RL_EXPORT int b200rl_hosttest_pack_weights_wide(const float* W1, const float* W2, const float* W3, const float* W_head, int D, int A, void* wpack) {
    using N = NetW;
    if (!net_is_wide(D, N::U1, N::U2, N::U3, A)) return B200RL_EUNSUPPORTED;
    const PackSeg seg[4] = {PackSeg{W1, N::U1, D, N::U1, N::DPAD, N::W1_OFF}, PackSeg{W2, N::U2, N::U1, N::U2, N::U1, N::W2_OFF},
                            PackSeg{W3, N::U3, N::U2, N::U3, N::U2, N::W3_OFF}, PackSeg{W_head, A + 1, N::U3, N::AP, N::U3, N::WH_OFF}};
    for (const PackSeg& s : seg) {
        const int ncg = s.Cpad / 8;
        const uint32_t CS = (uint32_t)(s.Rpad / 8) * 128u;
        for (int i = 0; i < s.Rpad * ncg; ++i) {
            const int r = i / ncg, cg = i - r * ncg;
            float f[8];
            for (int j = 0; j < 8; ++j) {
                const int c = cg * 8 + j;
                f[j] = (r < s.R && c < s.C) ? s.src[(size_t)r * s.C + c] : 0.f;
            }
            *reinterpret_cast<uint4*>((uint8_t*)wpack + s.dst_off + tile_off(r, cg, CS, 128u)) = pack8_bf16(f);
        }
    }
    return B200RL_OK;
}
#endif  // B200RL_TEST_HOOKS
#endif  // B200RL_TC_MAIN
