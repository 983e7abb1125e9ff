// drl_h256.cuh -- parameter layouts and constants of the 256-wide actor-critic (BASELINE config C5: the reference's
// ActorCritic of deep_rl/ppo.py:31-47 with hidden = 256 instead of 64).  At this width the two hidden layers are real
// contractions (2 x 256 x 256 MACs per net and sample), W2 alone is 128 KB in bf16 and its gradient fills the whole
// tensor memory of an SM, so the kernels differ from the 64-wide ones (update256.cu, rollout256.cu):
//   * one net per CTA (W2 of that net resident in shared memory for forward and backward),
//   * activations stream through four 16 KB K-chunks ([128 samples x 64 units] bf16, SW128),
//   * h1 and dz2 are staged in global memory (bf16, in the exact shared-memory image a 128-sample tile has), and a second
//     kernel -- a split-K tcgen05 GEMM -- turns them into dW2.
#pragma once
#include <cuda_bf16.h>

#include "drl_common.cuh"
#include "drl_tc_common.cuh"

namespace drl {
namespace h256 {

constexpr int HH = 256;              // hidden width
constexpr int NCH = 4;               // 64-unit chunks per layer
constexpr int SLOT_BYTES = 16384;    // one [128 x 64] bf16 SW128 chunk
constexpr int TILE_BYTES = NCH * SLOT_BYTES;   // one [128 x 256] activation tile (h1 or dz2) in its shared-memory image

// Packed (kernel) layout, in floats.  net 0 = actor, 1 = critic.
//   W2   : bf16 [2][4 chunks c][256 rows o][64 i]: SW128 K-major image, 16-byte unit u of row o stored at u ^ (o & 7)   (128 KB per net)
//   W1B  : bf16 [2][2 K-chunks][256 rows n][8]: K-major no-swizzle B operand of the layer-1 GEMM (K = 16):
//          k < O: W1[n][k], k == O: b1[n], k in [8, 8 + O): W1[n][k - 8] again (multiplies the low half of the observation)
//   B2   : fp32 [2][256]
//   W4   : fp32 [A + 1][256] (actor rows, then the critic row), B4 : fp32 [4] (actor biases, critic bias at [A])
//   W1F  : fp32 [2][256][OW] and B1F : fp32 [2][256], bf16-ROUNDED values (CUDA-core layer 1 of the rollout = the GEMM's operands)
template <int O, int A>
struct Packed256 {
    static constexpr int OW = O <= 4 ? 4 : 8;
    static constexpr int W2 = 0;
    static constexpr int W1B = W2 + 2 * HH * HH / 2;
    static constexpr int B2 = W1B + 2 * 2 * HH * 8 / 2;
    static constexpr int W4 = B2 + 2 * HH;
    static constexpr int B4 = W4 + (A + 1) * HH;
    static constexpr int W1F = B4 + 4;
    static constexpr int B1F = W1F + 2 * HH * OW;
    static constexpr int TOTAL = B1F + 2 * HH;
    // canonical (state_dict) layout
    static constexpr int C_NET = HH * O + HH + HH * HH + HH;      // trunk parameters per net
    static constexpr int C_ACTOR = C_NET + A * HH + A;
    static constexpr int C_ALL = C_ACTOR + C_NET + HH + 1;
    static constexpr int W2_OFF = HH * O + HH;                    // offset of W2 inside a net's canonical block
};

// byte offset of element (row o, column i) inside a net's W2 image
__host__ __device__ inline int w2_image_off(int o, int i) {
    const int c = i >> 6, u = (i & 63) >> 3;
    return c * (HH * 128) + o * 128 + ((u ^ (o & 7)) << 4) + (i & 7) * 2;
}

template <int O, int A>
__device__ __forceinline__ void packed_store256(float* __restrict__ packed, int idx, float v) {
    using P = Packed256<O, A>;
    const int net = idx >= P::C_ACTOR ? 1 : 0;
    int r = idx - net * P::C_ACTOR;
    const __nv_bfloat16 vb = __float2bfloat16_rn(v);
    if (r < HH * O) {
        const int o = r / O, k = r % O;
        __nv_bfloat16* w1b = reinterpret_cast<__nv_bfloat16*>(packed + P::W1B) + net * (2 * HH * 8);
        w1b[o * 8 + k] = vb;                  // K-chunk 0: multiplies obs_hi
        w1b[HH * 8 + o * 8 + k] = vb;         // K-chunk 1: multiplies obs_lo
        packed[P::W1F + (net * HH + o) * P::OW + k] = __bfloat162float(vb);
        return;
    }
    r -= HH * O;
    if (r < HH) {
        reinterpret_cast<__nv_bfloat16*>(packed + P::W1B)[net * (2 * HH * 8) + r * 8 + O] = vb;      // multiplies the ones column
        packed[P::B1F + net * HH + r] = __bfloat162float(vb);
        return;
    }
    r -= HH;
    if (r < HH * HH) {
        unsigned char* img = reinterpret_cast<unsigned char*>(packed + P::W2) + (size_t)net * (HH * HH * 2);
        *reinterpret_cast<__nv_bfloat16*>(img + w2_image_off(r / HH, r % HH)) = vb;
        return;
    }
    r -= HH * HH;
    if (r < HH) { packed[P::B2 + net * HH + r] = v; return; }
    r -= HH;
    const int nout = net == 0 ? A : 1;
    if (r < nout * HH) { packed[P::W4 + ((net == 0 ? 0 : A) + r / HH) * HH + r % HH] = v; return; }
    r -= nout * HH;
    packed[P::B4 + (net == 0 ? r : A)] = v;
}

// column of the [obs_hi | 1 | obs_lo] operand tile (16 columns) that carries output gradient `a` of the current net: the
// tile has free columns (their W1B rows are zero), so dW4 = h2^T . dout comes out of an N = 16 GEMM against the same tile
__host__ __device__ constexpr int dout_col(int O, int a) { return O <= 4 ? O + 1 + a : (a == 0 ? 7 : 13 + a); }

struct Grad256Args {
    const float* packed;
    const float* rec;          // [B][RW] sample records (gradient mode) or observations [n][OP] (forward mode)
    const uint32_t* idx;       // permutation (nullable)
    uint32_t mb_start, mb_count;      // this launch covers samples [mb_start, mb_start + mb_count) of the permuted order
    uint32_t mb_total;         // size of the whole minibatch (the mean's denominator)
    const float* adv_stats;
    float clip_coef, ent_coef, vf_coef;
    unsigned char* stage_h1;   // [2 nets][tiles][TILE_BYTES]
    unsigned char* stage_dz;
    uint32_t stage_tiles;      // tiles per net in the staging buffers
    float* grad_part;          // [grid][ppad], accumulated (read-modify-write, row owned by the CTA)
    float* loss_part;          // [grid][LOSS_TERMS], accumulated
    int ppad;
    float* logits_out;         // forward mode: [n][A]
    float* value_out;          // forward mode: [n]
    int only_net;              // -1: even CTAs the actor, odd CTAs the critic; 0 / 1: every CTA that net
    int first;                 // 1: first launch of this minibatch: the CTA WRITES its partial sums instead of adding to them
    long long* dbg;            // optional cycle stamps of CTA 0 (DRL_TC_DEBUG=1), else nullptr
};

constexpr int STAGE_TILES = 4096;   // 128-sample tiles per net the staging buffers hold (524,288 samples per pair of launches)

// ---- The actor's per-step forward pass on 128 envs, shared by rollout256_kernel (rollout256.cu) and evaluate256_kernel
// (eval256.cu).  Both kernels run these phases and nothing else between observation and logits, so they compute
// bit-identical logits for the same observation: a sampled evaluation replays what the training rollout would have done.
// Threads: 16 compute warps (warp w: row quarter q = w & 3, column quarter j = w >> 2; thread row r = 32 q + lane) and the
// MMA-issuer warp.  Named barriers (the issuer syncs, the 512 compute threads arrive):
enum : uint32_t { RB_H1 = 1, RB_L1 = 5, RB_QUAD = 6 };     // h1 chunk c ready (1..4), operand tile ready, row-quarter exchange (6..9)
constexpr uint32_t RB_ALL = TC_COMPUTE + 32;
constexpr uint32_t AF_Z1 = 0, AF_Z2 = 256;                 // TMEM columns of z1 and z2

template <int O, int A>
struct RoSmem256 {
    static constexpr int OFF_W2 = 0;
    static constexpr int OFF_ACT = OFF_W2 + HH * HH * 2;
    static constexpr int OFF_W1B = OFF_ACT + TILE_BYTES;
    static constexpr int OFF_B2 = OFF_W1B + 2 * HH * 8 * 2;
    static constexpr int OFF_W4 = OFF_B2 + HH * 4;
    static constexpr int OFF_B4 = OFF_W4 + 3 * HH * 4;
    static constexpr int OFF_OBS = OFF_B4 + 128;
    static constexpr int OFF_XCH = OFF_OBS + 4096;
    static constexpr int OFF_BAR = OFF_XCH + 4 * 3 * 128 * 4;
    static constexpr int TOTAL = OFF_BAR + 64 + 1024;
    static_assert(TOTAL <= 232448, "shared memory");
};

// S0 (owner threads): row r of the [obs_hi | 1 | obs_lo] operand tile of the K = 16 layer-1 GEMM
template <int O, int OP>
__device__ __forceinline__ void actor_l1_row(unsigned char* tOBS, int r, const float (&obs)[OP]) {
    float o16[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) o16[i] = 0.0f;
#pragma unroll
    for (int i = 0; i < O; ++i) {
        const float hi = __bfloat162float(__float2bfloat16_rn(obs[i]));
        o16[i] = hi;
        o16[8 + i] = obs[i] - hi;
    }
    o16[O] = 1.0f;
    umma::store_row_ns16(tOBS, TC_TILE, r, o16);
    umma::fence_proxy_async();
}

// Issuer warp, one step: the layer-1 GEMM once the operand tile is complete (RB_L1), then the layer-2 GEMM (M128 N256 K256)
// chunk by chunk as P0 completes the h1 chunks (RB_H1 + c).  Commits bars[1] after layer 1 and bars[2] after layer 2.
__device__ __forceinline__ void actor_issue_step(uint32_t tmem, uint32_t aOBS, uint32_t aW1B, uint32_t aACT, uint32_t aW2, uint64_t* bars) {
    constexpr uint32_t ID_L1 = umma::make_idesc(128, 256, false, false);
    constexpr uint32_t ID_FWD = umma::make_idesc(128, 256, false, false);
    named_bar_sync(RB_L1, RB_ALL);
    umma::fence_after_sync();
    if (umma::elect_one()) {
        umma::mma(tmem + AF_Z1, umma::make_desc(aOBS, 2048, 128, umma::LAYOUT_NONE),
                  umma::make_desc(aW1B, 4096, 128, umma::LAYOUT_NONE), ID_L1, 0u);
        umma::commit(bars + 1);
    }
    __syncwarp();
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
        named_bar_sync(RB_H1 + c, RB_ALL);
        umma::fence_after_sync();
        if (umma::elect_one()) {
#pragma unroll
            for (int kb = 0; kb < 4; ++kb)
                umma::mma(tmem + AF_Z2, umma::make_desc(aACT + c * SLOT_BYTES + kb * 32, 16, 1024, umma::LAYOUT_SW128),
                          umma::make_desc(aW2 + c * 32768 + kb * 32, 16, 1024, umma::LAYOUT_SW128), ID_FWD, (c > 0 || kb > 0) ? 1u : 0u);
            if (c == NCH - 1) umma::commit(bars + 2);
        }
        __syncwarp();
    }
}

// P0 (all compute threads): wait for layer 1, h1 = tanh(z1) -> four bf16 K-chunks of the layer-2 A operand; each chunk is
// released to the issuer as soon as it is written.  `parity` = phase of bars[1] (step & 1).
__device__ __forceinline__ void actor_h1_chunks(uint32_t trow, unsigned char* tACT, uint32_t off0, uint32_t off1, int j, uint64_t* bars,
                                                uint32_t parity) {
    mbar_wait(bars + 1, parity);
    umma::fence_after_sync();
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
        float z[16];
        umma::ld16(trow + AF_Z1 + 64 * c + 16 * j, z);
#pragma unroll
        for (int x = 0; x < 16; ++x) z[x] = tanh_mufu(z[x]);
        uint4 q0, q1;
        q0.x = umma::pack_bf16(z[0], z[1]); q0.y = umma::pack_bf16(z[2], z[3]); q0.z = umma::pack_bf16(z[4], z[5]); q0.w = umma::pack_bf16(z[6], z[7]);
        q1.x = umma::pack_bf16(z[8], z[9]); q1.y = umma::pack_bf16(z[10], z[11]); q1.z = umma::pack_bf16(z[12], z[13]); q1.w = umma::pack_bf16(z[14], z[15]);
        *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off0) = q0;
        *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off1) = q1;
        umma::fence_proxy_async();
        umma::fence_before_sync();
        named_bar_arrive(RB_H1 + c, RB_ALL);
    }
}

// P1 (all compute threads): wait for layer 2, h2 = tanh(z2 + b2) on this thread's 64 units, partial head sums -> xch
// (the caller makes them visible to its row quarter with RB_QUAD + q).  `parity` = phase of bars[2] (step & 1).
template <int A>
__device__ __forceinline__ void actor_head_partials(uint32_t trow, const float* sB2, const float* sW4, float* xch, int j, int r,
                                                    uint64_t* bars, uint32_t parity) {
    mbar_wait(bars + 2, parity);
    umma::fence_after_sync();
    float ps[A];
#pragma unroll
    for (int a = 0; a < A; ++a) ps[a] = 0.0f;
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
        float z[16];
        umma::ld16(trow + AF_Z2 + 64 * c + 16 * j, z);
#pragma unroll
        for (int e4 = 0; e4 < 4; ++e4) {
            const float4 bb = *reinterpret_cast<const float4*>(sB2 + 64 * c + 16 * j + 4 * e4);
            z[4 * e4 + 0] = tanh_mufu(z[4 * e4 + 0] + bb.x);
            z[4 * e4 + 1] = tanh_mufu(z[4 * e4 + 1] + bb.y);
            z[4 * e4 + 2] = tanh_mufu(z[4 * e4 + 2] + bb.z);
            z[4 * e4 + 3] = tanh_mufu(z[4 * e4 + 3] + bb.w);
        }
#pragma unroll
        for (int a = 0; a < A; ++a) {
            const float* w = sW4 + a * HH + 64 * c + 16 * j;
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
                const float4 ww = *reinterpret_cast<const float4*>(w + 4 * e4);
                s0 = fmaf(z[4 * e4 + 0], ww.x, s0);
                s1 = fmaf(z[4 * e4 + 1], ww.y, s1);
                s2 = fmaf(z[4 * e4 + 2], ww.z, s2);
                s3 = fmaf(z[4 * e4 + 3], ww.w, s3);
            }
            ps[a] += (s0 + s1) + (s2 + s3);
        }
    }
#pragma unroll
    for (int a = 0; a < A; ++a) xch[(j * 3 + a) * TC_TILE + r] = ps[a];
}

// S3 (owner threads, after the exchange barrier): the logits of row r, summed in a fixed order over the four column quarters
template <int A>
__device__ __forceinline__ void actor_logits(const float* xch, const float* sB4, int r, float (&l)[A]) {
#pragma unroll
    for (int a = 0; a < A; ++a)
        l[a] = ((xch[(0 * 3 + a) * TC_TILE + r] + xch[(1 * 3 + a) * TC_TILE + r]) +
                (xch[(2 * 3 + a) * TC_TILE + r] + xch[(3 * 3 + a) * TC_TILE + r])) + sB4[a];
}

}  // namespace h256
}  // namespace drl
