// drl_common.cuh -- shared device/host helpers for libdrl_b200 (sm_100a only).
// Compiled with -fmad=false: every fused multiply-add in this library is an explicit fmaf()/fma(),
// so the op-order-sensitive pieces (GAE, sampler, env physics, reset draws) round exactly like the
// reference's eager fp32/fp64 arithmetic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/drl_b200.h"

namespace drl {

// ----------------------------------------------------------------------------------------------
// error plumbing (no exceptions across the C ABI)
// ----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define DRL_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            drl::set_error(__VA_ARGS__);       \
            return DRL_ERR_ARG;                \
        }                                      \
    } while (0)

#define DRL_CUDA(call)                                             \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return drl::cuda_fail(e__, #call); \
    } while (0)

#define DRL_LAUNCH_CHECK(name)                                      \
    do {                                                            \
        cudaError_t e__ = cudaPeekAtLastError();                    \
        if (e__ != cudaSuccess) return drl::cuda_fail(e__, name);   \
    } while (0)

int sm_count();

// ----------------------------------------------------------------------------------------------
// network geometry.  H is fixed at 64 in this build: a warp owns an 8-sample tile, its two
// half-warps own the actor / critic trunk, each lane owns UPL = H/16 = 4 hidden units.
// ----------------------------------------------------------------------------------------------
constexpr int H = 64;
constexpr int TILE = 8;   // samples (envs) per warp tile
constexpr int UPL = 4;    // hidden units per lane

// lane-permuted position of hidden unit `unit`: lane u = unit & 15 owns positions 4u..4u+3,
// position 4u+j <-> unit u + 16j.  Consecutive lanes then store consecutive rows of the
// activation tile (conflict-free) while their four weights stay one 16-byte load.
__host__ __device__ constexpr int perm_pos(int unit) { return 4 * (unit & 15) + (unit >> 4); }

// Packed (kernel) parameter layout, in floats.  net 0 = actor, net 1 = critic.
//   W1T[2][O][H]  : W1T[net][i][perm_pos(o)] = W1[o][i]
//   b1 [2][H]     : permuted
//   W2T[2][H][H]  : W2T[net][k][perm_pos(o)] = W2[o][k]          (forward:  z2 = h1 . W2^T)
//   b2 [2][H]     : permuted
//   W4 [2][A][H]  : W4[net][a][perm_pos(k)] = Whead[a][k]; critic uses row 0, other rows stay 0
//   b4 [2][A]     : critic uses slot 0
//   ---- forward kernels stage up to here (fwd_count) ----
//   W2P[2][H][H]  : W2P[net][o][perm_pos(i)] = W2[o][i]          (backward: dh1 = dz2 . W2)
template <int O, int A>
struct Packed {
    static constexpr int W1T = 0;
    static constexpr int B1 = W1T + 2 * O * H;
    static constexpr int W2T = B1 + 2 * H;
    static constexpr int B2 = W2T + 2 * H * H;
    static constexpr int W4 = B2 + 2 * H;
    static constexpr int B4 = W4 + 2 * A * H;
    static constexpr int FWD_RAW = B4 + 2 * A;
    static constexpr int FWD = (FWD_RAW + 3) / 4 * 4;  // 16-byte multiple for the bulk copy
    static constexpr int W2P = FWD;
    static constexpr int ALL = W2P + 2 * H * H;
    // ---- tensor-core section (update_tc.cu), natural unit order, staged by one TMA bulk copy ----
    //   TC_W2 : bf16 [2][64 rows o][64 i] as two SW128 UMMA tiles (16 KB)
    //   TC_W1 : fp32 [2][H][OW] (OW = 4 or 8, zero padded) and TC_B1 : fp32 [2][H], both holding bf16-ROUNDED values (the
    //           rollout's CUDA-core layer 1 then matches the update's layer-1 GEMM operands); TC_B2 : fp32 [2][H]
    //   TC_W4 : fp32 [A+1][H] (actor rows, then the critic row), TC_B4 : fp32 [4]
    static constexpr int OW = O <= 4 ? 4 : 8;
    static constexpr int TC_W2 = ALL;
    static constexpr int TC_W1 = TC_W2 + 2 * H * H / 2;
    static constexpr int TC_B1 = TC_W1 + 2 * H * OW;
    static constexpr int TC_B2 = TC_B1 + 2 * H;
    static constexpr int TC_W4 = TC_B2 + 2 * H;
    static constexpr int TC_B4 = TC_W4 + (A + 1) * H;
    //   TC_W1B: bf16 [2][2 chunks][H rows][8]: K-major no-swizzle B operand of the layer-1 GEMM, K = 16:
    //           k < O: W1[n][k], k == O: b1[n], k in [8, 8+O): W1[n][k-8] again (multiplies the low half of obs)
    static constexpr int TC_W1B = TC_B4 + 4;
    static constexpr int TC_END = TC_W1B + 2 * 2 * H * 8 / 2;
    static constexpr int TOTAL = TC_END;
    // canonical (state_dict) layout
    static constexpr int C_NET = H * O + H + H * H + H;          // trunk params per net
    static constexpr int C_ACTOR = C_NET + A * H + A;
    static constexpr int C_ALL = C_ACTOR + C_NET + H + 1;
};

// ----------------------------------------------------------------------------------------------
// Philox4x32-10; stream definition mirrors oracle/drl_oracle.c (the RNG contract of this build).
// ----------------------------------------------------------------------------------------------
enum : uint32_t { TAG_ACTION = 0, TAG_RESET = 1, TAG_PERM = 2 };

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint4 philox_seeded(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
    return philox4x32_10(c0, c1, c2, c3, (uint32_t)seed, (uint32_t)(seed >> 32));
}

__device__ __forceinline__ float u01_f32(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }
__device__ __forceinline__ double u01_f64(uint32_t x) { return ((double)x + 0.5) * 2.3283064365386963e-10; }

// Deterministic expf for the sampler: IEEE ops + explicit fmaf only -> bit-identical to the oracle.
__device__ __forceinline__ float exp_det(float x) {
    if (x < -87.0f) return 0.0f;
    if (x > 88.0f) x = 88.0f;
    float t = __fmul_rn(x, 1.44269504088896341f);
    float n = rintf(t);
    float r = __fmaf_rn(n, -0.693145751953125f, x);
    r = __fmaf_rn(n, -1.428606765330187045e-06f, r);
    float p = 1.9875691500e-4f;
    p = __fmaf_rn(p, r, 1.3981999507e-3f);
    p = __fmaf_rn(p, r, 8.3334519073e-3f);
    p = __fmaf_rn(p, r, 4.1665795894e-2f);
    p = __fmaf_rn(p, r, 1.6666665459e-1f);
    p = __fmaf_rn(p, r, 5.0000001201e-1f);
    float r2 = __fmul_rn(r, r);
    float e = __fmaf_rn(p, r2, r);
    e = __fadd_rn(e, 1.0f);
    int ni = (int)n;
    float s = __uint_as_float((uint32_t)(ni + 127) << 23);
    return __fmul_rn(e, s);
}

// Inverse-CDF categorical draw (mirrored bit-for-bit by the CPU oracle).  Returns the action and the
// log-probability (l_act - max) - log(sum).
template <int A>
__device__ __forceinline__ int sample_categorical(const float (&l)[A], float u, float& logp) {
    float m = l[0];
#pragma unroll
    for (int a = 1; a < A; ++a) m = l[a] > m ? l[a] : m;
    float e[A];
    float s = 0.0f;
#pragma unroll
    for (int a = 0; a < A; ++a) { e[a] = exp_det(__fsub_rn(l[a], m)); s = __fadd_rn(s, e[a]); }
    float thr = __fmul_rn(u, s);
    float c = 0.0f;
    int act = A - 1;
    bool found = false;
    float lsel = l[A - 1];
#pragma unroll
    for (int a = 0; a < A - 1; ++a) {
        c = __fadd_rn(c, e[a]);
        if (!found && thr < c) { act = a; lsel = l[a]; found = true; }
    }
    logp = __fsub_rn(__fsub_rn(lsel, m), logf(s));
    return act;
}

// first index of the largest logit (the torch.argmax tie rule)
template <int A>
__device__ __forceinline__ int argmax_first(const float (&l)[A]) {
    int best = 0;
    float m = l[0];
#pragma unroll
    for (int a = 1; a < A; ++a)
        if (l[a] > m) { m = l[a]; best = a; }
    return best;
}

// The same draw with the log-probability left in two pieces, logp = diff - logf(sum): the fused rollout finishes it off the
// critical path of the step.  Bit-identical to sample_categorical.
template <int A>
__device__ __forceinline__ int sample_categorical_split(const float (&l)[A], float u, float& diff, float& sum) {
    float m = l[0];
#pragma unroll
    for (int a = 1; a < A; ++a) m = l[a] > m ? l[a] : m;
    float e[A];
    float s = 0.0f;
#pragma unroll
    for (int a = 0; a < A; ++a) { e[a] = exp_det(__fsub_rn(l[a], m)); s = __fadd_rn(s, e[a]); }
    float thr = __fmul_rn(u, s);
    float c = 0.0f;
    int act = A - 1;
    bool found = false;
    float lsel = l[A - 1];
#pragma unroll
    for (int a = 0; a < A - 1; ++a) {
        c = __fadd_rn(c, e[a]);
        if (!found && thr < c) { act = a; lsel = l[a]; found = true; }
    }
    diff = __fsub_rn(lsel, m);
    sum = s;
    return act;
}

// tanh with two MUFU ops (ex2, rcp): |abs err| ~ 2e-7; saturates correctly at +-1.
__device__ __forceinline__ float tanh_fast(float x) {
    float t, r;
    float y = x * 2.885390081777927f;  // 2*log2(e)
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(y));
    float d = t + 1.0f;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
    return fmaf(-2.0f, r, 1.0f);
}

// ----------------------------------------------------------------------------------------------
// shared-memory / TMA bulk-copy helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {   // release at CTA scope: prior st.shared of this thread are ordered before it
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
// 1-D TMA bulk copy global -> shared (SASS: UBLKCP); bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// 1-D TMA bulk copy shared -> global (bulk async-group completion).  The shared-memory source must have been made visible to the
// async proxy (fence.proxy.async by its writers, then a barrier) before the issuing thread executes this.
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all bulk groups of this thread have finished READING their shared-memory sources (the sources may be overwritten)
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all bulk groups of this thread have completed (their global writes are performed)
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Stage `nfloats` (multiple of 4) of packed parameters into shared memory with TMA bulk copies issued
// by thread 0; every thread returns once the bytes have landed.  `bar` is a shared mbarrier slot.
__device__ __forceinline__ void stage_params(float* dst, const float* __restrict__ src, int nfloats, uint64_t* bar) {
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t total = (uint32_t)nfloats * 4u;
        mbar_expect_tx(bar, total);
        constexpr uint32_t CHUNK = 32768u;
        for (uint32_t off = 0; off < total; off += CHUNK) {
            uint32_t n = total - off < CHUNK ? total - off : CHUNK;
            bulk_g2s((char*)dst + off, (const char*)src + off, n, bar);
        }
    }
    mbar_wait(bar, 0);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

inline cudaStream_t as_stream(void* s) { return (cudaStream_t)s; }

}  // namespace drl
