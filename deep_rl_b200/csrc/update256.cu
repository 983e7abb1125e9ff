// update256.cu -- PPO minibatch gradient (deep_rl/ppo.py:159-190) and batched forward (ppo.py:49-54) for the 256-wide
// actor-critic (BASELINE config C5) on tcgen05 tensor cores.  Two kernels per chunk of samples:
//
//   mlp256_kernel      persistent, one CTA per SM, ONE NET per CTA (even CTAs the actor, odd CTAs the critic; the 128 KB bf16
//                      image of that net's W2 stays in shared memory for the forward and the backward pass), 128-sample tiles:
//        L1    z1 = [obs_hi|1|obs_lo] . [W1|b1|W1]^T            one M128 N256 K16 MMA
//        P0    h1 = tanh(z1) -> four bf16 K-chunks [128 x 64] in a shared-memory ring AND in the global staging buffer
//        fwd   z2 = h1 . W2^T, issued K-chunk by K-chunk as P0 produces them, in two N-halves (128 TMEM columns)
//        P1    h2 = tanh(z2 + b2), heads, loss and closed-form output gradients; h2 -> ring -> dW4 += h2^T . dout (N = 16)
//              dz2 = (dout . W4) * (1 - h2^2) -> ring + staging
//        bwd   dh1 = dz2 . W2 (same W2 image, MN-major descriptor), K-chunk by K-chunk; db2 += dz2^T . 1 (N = 16)
//        P2    dz1 = dh1 * (1 - h1^2) -> ring -> [dW1|db1] += dz1^T . [obs|1] (N = 16)
//      The small weight-gradient accumulators (96 TMEM columns) live in tensor memory for the whole kernel; dW2 does not fit
//      (256 x 256 fp32 = all 512 columns), hence:
//   dw2_gemm256_kernel split-K GEMM dW2 = dz2^T . h1 over the staged tiles: TMA bulk copies (the staging buffer holds the exact
//                      SW128 shared-memory image of every tile, so plain 1-D copies suffice) into a 3-stage ring, two
//                      M128 N256 K16 MMAs per 16 samples, the full 512-column accumulator, one pass over the data.
// Both kernels ADD their per-CTA partial sums to row blockIdx.x of the partial-gradient buffer (zeroed once per minibatch by the
// launcher); grad_reduce_kernel then folds the rows in a fixed order, exactly as on the 64-wide path.
#include "drl_h256.cuh"
#include "drl_pack.cuh"
#include "drl_tc_common.cuh"
#include "drl_update.cuh"

namespace drl {
namespace h256 {

// tensor-memory columns: z2 halves, then (with C_X) the 256 columns of dh1 | z1 halves | packed bf16 h1 stash | small accumulators
constexpr uint32_t C_Z2 = 0, C_X = 128, C_DH = 0, C_H1P = 256, C_SW4 = 416, C_SW1 = 448, TM_COLS = 512;
constexpr int A_BLOCK = TC_COMPUTE + 64;   // 16 compute warps + MMA-issuer warp + loader warp
constexpr int OBS_RING = 2;

// named barriers (0 = __syncthreads)
enum : uint32_t { NB_H1 = 1, NB_DZ2 = 5, NB_Z2A = 9, NB_W4RDY = 10, NB_DZ1 = 11, NB_QUAD = 12 };
constexpr uint32_t NB_ALL = TC_COMPUTE + 32;    // compute threads arrive, the issuer warp syncs

template <int O, int A>
struct Smem256 {
    static constexpr int OFF_W2 = 0;                                   // 128 KB
    static constexpr int OFF_ACT = OFF_W2 + HH * HH * 2;               // four 16 KB chunks
    static constexpr int OFF_W1B = OFF_ACT + TILE_BYTES;               // 8 KB
    static constexpr int OFF_B2 = OFF_W1B + 2 * HH * 8 * 2;            // 1 KB
    static constexpr int OFF_W4 = OFF_B2 + HH * 4;                     // up to 3 rows
    static constexpr int OFF_B4 = OFF_W4 + 3 * HH * 4;
    static constexpr int OFF_OBS = OFF_B4 + 128;                       // two NS16 tiles [obs_hi|1|obs_lo]
    static constexpr int OFF_SCAL = OFF_OBS + OBS_RING * 4096;         // two buffers of per-row scalars
    static constexpr int OFF_XCH = OFF_SCAL + OBS_RING * 2048;         // head partial sums [4 column blocks][3 heads][128 rows]
    static constexpr int OFF_BAR = OFF_XCH + 4 * 3 * 128 * 4;
    static constexpr int OFF_RED = OFF_BAR + 256;
    static constexpr int TOTAL = OFF_RED + 16 * 12 * 4 + 1024;
    static_assert(TOTAL <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
    static_assert(OFF_OBS % 128 == 0, "operand tile alignment");
};

// diagnostics: cycle stamps of CTA 0, compute warp 0 (slot = tile * 16 + event) and issuer warp (256 + ...), DRL_TC_DEBUG=1
#define H2_STAMP(ev) do { if (g.dbg != nullptr && blockIdx.x == 0 && lane == 0 && k < 8 && (warp == 0 || warp == TC_COMPUTE / 32)) g.dbg[(warp == 0 ? 0 : 256) + k * 16 + (ev)] = clock64(); } while (0)

// MODE 0: gradient (records in, partial gradients out); MODE 1: forward only (observations in, logits / values out)
template <int O, int A, int OP, int RW, int MODE>
__global__ void __launch_bounds__(A_BLOCK, 1) mlp256_kernel(Grad256Args g) {
    using P = Packed256<O, A>;
    using S = Smem256<O, A>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* tW2 = sm + S::OFF_W2;
    unsigned char* tACT = sm + S::OFF_ACT;
    unsigned char* tW1B = sm + S::OFF_W1B;
    const float* sB2 = reinterpret_cast<const float*>(sm + S::OFF_B2);
    const float* sW4 = reinterpret_cast<const float*>(sm + S::OFF_W4);
    const float* sB4 = reinterpret_cast<const float*>(sm + S::OFF_B4);
    unsigned char* tOBS = sm + S::OFF_OBS;
    uint4* sSCAL = reinterpret_cast<uint4*>(sm + S::OFF_SCAL);
    float* xch = reinterpret_cast<float*>(sm + S::OFF_XCH);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + S::OFF_BAR);   // 0 weights, 1 l1 (units 0..127), 2 fwd-a, 3 fwd-b, 4 dW4, 5 dh1+db2, 6 dW1, 7 l1 (units 128..255)
    uint64_t* ring_full = bars + 8;
    uint64_t* ring_empty = bars + 8 + OBS_RING;
    uint32_t* slot = reinterpret_cast<uint32_t*>(bars + 8 + 2 * OBS_RING);
    float* red = reinterpret_cast<float*>(sm + S::OFF_RED);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool is_mma_warp = warp == TC_COMPUTE / 32;
    const bool is_loader_warp = warp == TC_COMPUTE / 32 + 1;
    const int net = g.only_net >= 0 ? g.only_net : (int)(blockIdx.x & 1);
    const uint32_t cin = g.only_net >= 0 ? blockIdx.x : blockIdx.x >> 1;  // this CTA among the CTAs of its net
    const uint32_t ncn = g.only_net >= 0 ? gridDim.x : gridDim.x >> 1;
    const uint32_t ntiles = (g.mb_count + TC_TILE - 1) / TC_TILE;
    if (cin >= ntiles) return;                                            // nothing to do (uniform for the whole CTA)
    const uint32_t nmy = (ntiles - cin + ncn - 1) / ncn;
    constexpr int nheads_a = A;
    const int nheads = net == 0 ? nheads_a : 1;

    // ---- prologue ----
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) mbar_init(bars + i, 1);
#pragma unroll
        for (int i = 0; i < OBS_RING; ++i) { mbar_init(ring_full + i, 32); mbar_init(ring_empty + i, 1); }
        mbar_fence_init();
    }
    if (warp == 1) umma::tmem_alloc(slot, TM_COLS);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    if (tid == 0) {
        const uint32_t w4_bytes = (uint32_t)nheads * HH * 4;
        mbar_expect_tx(bars, (uint32_t)(HH * HH * 2 + 2 * HH * 8 * 2 + HH * 4) + w4_bytes + 16u);
        const char* w2 = reinterpret_cast<const char*>(g.packed + P::W2) + (size_t)net * (HH * HH * 2);
        for (uint32_t off = 0; off < (uint32_t)(HH * HH * 2); off += 32768u) bulk_g2s(tW2 + off, w2 + off, 32768u, bars);
        bulk_g2s(tW1B, reinterpret_cast<const char*>(g.packed + P::W1B) + (size_t)net * (2 * HH * 8 * 2), 2 * HH * 8 * 2, bars);
        bulk_g2s(sm + S::OFF_B2, g.packed + P::B2 + net * HH, HH * 4, bars);
        bulk_g2s(sm + S::OFF_W4, g.packed + P::W4 + (net == 0 ? 0 : A) * HH, w4_bytes, bars);
        bulk_g2s(sm + S::OFF_B4, g.packed + P::B4, 16u, bars);
    }
    const uint32_t tmem = *slot;

    if (is_loader_warp) {
        // =========================== loader warp: lane l owns rows l, l+32, l+64, l+96 of every tile ===========================
        for (uint32_t j = 0; j < nmy; ++j) {
            const uint32_t tile = cin + j * ncn;
            const uint32_t b = j & 1u;
            float4 rv[4][OP / 4 + 1];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
#pragma unroll
                for (int c = 0; c <= OP / 4; ++c) rv[q][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                rv[q][OP / 4].w = __int_as_float(-1);                     // act < 0 marks a padding row
                const uint32_t pos = tile * TC_TILE + (uint32_t)(lane + 32 * q);
                if (pos < g.mb_count) {
                    const uint32_t i = g.mb_start + pos;
                    if (MODE == 0) {
                        const uint32_t s = g.idx ? __ldg(g.idx + i) : i;
                        const float4* r4 = reinterpret_cast<const float4*>(g.rec + (size_t)s * RW);
#pragma unroll
                        for (int c = 0; c < OP / 4; ++c) rv[q][c] = __ldg(r4 + c);
                        rv[q][OP / 4] = __ldg(r4 + RW / 4 - 1);
                    } else {
                        const float4* r4 = reinterpret_cast<const float4*>(g.rec + (size_t)i * OP);
#pragma unroll
                        for (int c = 0; c < OP / 4; ++c) rv[q][c] = __ldg(r4 + c);
                        rv[q][OP / 4].w = __int_as_float(0);
                    }
                }
            }
            if (j >= OBS_RING) mbar_wait(ring_empty + b, ((j >> 1) - 1u) & 1u);   // the GEMMs of tile j - 2 have released the slot
            unsigned char* obst = tOBS + b * 4096;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int row = lane + 32 * q;
                float o16[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) o16[i] = 0.0f;
#pragma unroll
                for (int i = 0; i < O; ++i) {
                    const float4 v4 = rv[q][i / 4];
                    const float x = (i & 3) == 0 ? v4.x : ((i & 3) == 1 ? v4.y : ((i & 3) == 2 ? v4.z : v4.w));
                    const float hi = __bfloat162float(__float2bfloat16_rn(x));
                    o16[i] = hi;
                    o16[8 + i] = x - hi;
                }
                o16[O] = 1.0f;
                umma::store_row_ns16(obst, TC_TILE, row, o16);
                sSCAL[b * TC_TILE + row] = make_uint4(__float_as_uint(rv[q][OP / 4].x), __float_as_uint(rv[q][OP / 4].y),
                                                      __float_as_uint(rv[q][OP / 4].z), __float_as_uint(rv[q][OP / 4].w));
            }
            umma::fence_proxy_async();
            mbar_arrive(ring_full + b);
        }
        __syncthreads();
        return;
    }

    if (is_mma_warp) {
        // =========================== MMA-issuer warp ===========================
        const uint32_t aW2 = smem_u32(tW2), aACT = smem_u32(tACT), aW1B = smem_u32(tW1B), aOBS = smem_u32(tOBS);
        constexpr uint32_t ID_L1 = umma::make_idesc(128, 128, false, false);
        constexpr uint32_t ID_FWD = umma::make_idesc(128, 128, false, false);
        constexpr uint32_t ID_DH1 = umma::make_idesc(128, 256, false, true);
        constexpr uint32_t ID_N16 = umma::make_idesc(128, 16, true, true);
        mbar_wait(bars, 0);
        // layer 1, K = 16, no swizzle: A = operand tile, B = [W1|b1|W1]; units 0..127 first.  Issued for tile k + 1 as soon as the
        // upper half of the dh1 columns (which it overwrites) has been read in P2 of tile k.
        auto issue_l1a = [&](uint32_t kk) {
            const uint32_t bb = kk & 1u;
            mbar_wait(ring_full + bb, (kk >> 1) & 1u);
            umma::fence_after_sync();
            if (umma::elect_one()) {
                umma::mma(tmem + C_X, umma::make_desc(aOBS + bb * 4096, 2048, 128, umma::LAYOUT_NONE),
                          umma::make_desc(aW1B, 4096, 128, umma::LAYOUT_NONE), ID_L1, 0u);
                umma::commit(bars + 1);
            }
            __syncwarp();
        };
        issue_l1a(0);
        for (uint32_t k = 0; k < nmy; ++k) {
            const uint32_t b = k & 1u, acc = k > 0 ? 1u : 0u;
            const uint32_t obsb = aOBS + b * 4096;
            const uint32_t tile = cin + k * ncn;
            unsigned char* st_h1 = g.stage_h1 + ((size_t)net * g.stage_tiles + tile) * TILE_BYTES;
            unsigned char* st_dz = g.stage_dz + ((size_t)net * g.stage_tiles + tile) * TILE_BYTES;
            // forward, first N-half (units 0..127), K-chunk by K-chunk as the h1 chunks arrive
#pragma unroll 1
            for (int c = 0; c < NCH; ++c) {
                if (c == 0) {       // z1 of units 0..127 is in registers: layer 1 of units 128..255 into the same 128 columns
                    named_bar_sync(NB_Z2A, NB_ALL);
                    umma::fence_after_sync();
                    if (umma::elect_one()) {
                        umma::mma(tmem + C_X, umma::make_desc(obsb, 2048, 128, umma::LAYOUT_NONE),
                                  umma::make_desc(aW1B + 128 * 16, 4096, 128, umma::LAYOUT_NONE), ID_L1, 0u);
                        umma::commit(bars + 7);
                    }
                    __syncwarp();
                }
                named_bar_sync(NB_H1 + c, NB_ALL);
                umma::fence_after_sync();
                if (umma::elect_one()) {
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb)
                        umma::mma(tmem + C_Z2, umma::make_desc(aACT + c * SLOT_BYTES + kb * 32, 16, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(aW2 + c * 32768 + kb * 32, 16, 1024, umma::LAYOUT_SW128), ID_FWD, (c > 0 || kb > 0) ? 1u : 0u);
                    if (c == NCH - 1) umma::commit(bars + 2);
                }
                // the chunk is also what dw2_gemm256_kernel reads: one TMA bulk store of its 16 KB shared-memory image
                if (MODE == 0 && lane == 0) { bulk_s2g(st_h1 + c * SLOT_BYTES, tACT + c * SLOT_BYTES, SLOT_BYTES); bulk_commit_group(); }
                __syncwarp();
            }
            // forward, second N-half (units 128..255): the first half has been read out of tensor memory
            named_bar_sync(NB_Z2A, NB_ALL);
            umma::fence_after_sync();
            if (MODE == 0 && lane == 0) bulk_wait_group0();      // staged h1 complete: the ring is rewritten and the staging copy re-read
            __syncwarp();                                        // only after the commit below has fired
            if (umma::elect_one()) {
#pragma unroll 1
                for (int c = 0; c < NCH; ++c)
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb)
                        umma::mma(tmem + C_Z2, umma::make_desc(aACT + c * SLOT_BYTES + kb * 32, 16, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(aW2 + c * 32768 + 128 * 128 + kb * 32, 16, 1024, umma::LAYOUT_SW128), ID_FWD,
                                  (c > 0 || kb > 0) ? 1u : 0u);
                umma::commit(bars + 3);
            }
            __syncwarp();
            if (MODE == 1) {
                if (umma::elect_one()) umma::commit(ring_empty + b);
                __syncwarp();
                if (k + 1 < nmy) issue_l1a(k + 1);       // z1 of this tile was read long ago
                continue;
            }
            // dW4 += h2^T . dout   (h2 chunks in the ring, dout in the free columns of the operand tile)
            named_bar_sync(NB_W4RDY, NB_ALL);
            umma::fence_after_sync();
            if (umma::elect_one()) {
#pragma unroll
                for (int u = 0; u < 2; ++u)
#pragma unroll
                    for (int kb = 0; kb < 8; ++kb)
                        umma::mma(tmem + C_SW4 + 16 * u, umma::make_desc(aACT + u * 2 * SLOT_BYTES + kb * 2048, SLOT_BYTES, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(obsb + kb * 256, 128, 2048, umma::LAYOUT_NONE), ID_N16, acc | (kb > 0 ? 1u : 0u));
                umma::commit(bars + 4);
            }
            __syncwarp();
            // dh1 = dz2 . W2, K-chunk (64 units o) by K-chunk; B = the W2 image read MN-major (N = i: four 64-wide atoms)
#pragma unroll 1
            for (int c = 0; c < NCH; ++c) {
                named_bar_sync(NB_DZ2 + c, NB_ALL);
                umma::fence_after_sync();
                if (umma::elect_one()) {
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb)
                        umma::mma(tmem + C_DH, umma::make_desc(aACT + c * SLOT_BYTES + kb * 32, 16, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(aW2 + (4 * c + kb) * 2048, 32768, 1024, umma::LAYOUT_SW128), ID_DH1, (c > 0 || kb > 0) ? 1u : 0u);
                }
                if (lane == 0) { bulk_s2g(st_dz + c * SLOT_BYTES, tACT + c * SLOT_BYTES, SLOT_BYTES); bulk_commit_group(); }
                __syncwarp();
            }
            if (lane == 0) bulk_wait_group_read0();      // the staged dz2 chunks have been read out of the ring (P2 overwrites it)
            __syncwarp();
            if (umma::elect_one()) umma::commit(bars + 5);      // dh1 complete (db2 = column sums of dz2 comes from dw2_gemm256_kernel)
            __syncwarp();
            if (k + 1 < nmy) {       // dh1 columns 128..255 are in registers: layer 1 of the next tile may overwrite them
                named_bar_sync(NB_Z2A, NB_ALL);
                issue_l1a(k + 1);
            }
            // [dW1|db1] += dz1^T . [obs|1]
            named_bar_sync(NB_DZ1, NB_ALL);
            umma::fence_after_sync();
            if (umma::elect_one()) {
#pragma unroll
                for (int u = 0; u < 2; ++u)
#pragma unroll
                    for (int kb = 0; kb < 8; ++kb)
                        umma::mma(tmem + C_SW1 + 16 * u, umma::make_desc(aACT + u * 2 * SLOT_BYTES + kb * 2048, SLOT_BYTES, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(obsb + kb * 256, 128, 2048, umma::LAYOUT_NONE), ID_N16, acc | (kb > 0 ? 1u : 0u));
                umma::commit(bars + 6);
                umma::commit(ring_empty + b);
            }
            __syncwarp();
        }
        umma::fence_before_sync();
        __syncthreads();
        return;
    }

    // =========================== compute warps ===========================
    // warp w: TMEM lane quadrant q = w & 3 (rows 32q .. 32q+31), column block j = w >> 2: columns 64c + 16j .. +16 of every chunk c
    const int q = warp & 3, j = warp >> 2;
    const int r = q * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
    const float adv_mean = MODE == 0 ? g.adv_stats[0] : 0.0f, adv_rstd = MODE == 0 ? 1.0f / (g.adv_stats[1] + 1e-8f) : 0.0f;
    const float inv_m = 1.0f / (float)g.mb_total;
    float lsum[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    float gb4[3] = {0.f, 0.f, 0.f};
    mbar_wait(bars, 0);

    for (uint32_t k = 0; k < nmy; ++k) {
        const uint32_t par = k & 1u, b = k & 1u;
        const uint32_t tile = cin + k * ncn;
        const uint32_t off0 = umma::sw128_off(r, 2 * j), off1 = umma::sw128_off(r, 2 * j + 1);     // this thread's two 16-byte units of a chunk row

        // ================= P0: h1 = tanh(z1), chunk by chunk (z1 arrives in two halves of 128 units) =================
        H2_STAMP(0);
        mbar_wait(bars + 1, par);
        umma::fence_after_sync();
        H2_STAMP(1);
        float zz[2][16];
        umma::ld16(trow + C_X + 16 * j, zz[0]);
        umma::ld16(trow + C_X + 64 + 16 * j, zz[1]);
        umma::fence_before_sync();
        named_bar_arrive(NB_Z2A, NB_ALL);          // z1 of units 0..127 is in registers (the barrier is free until the forward GEMM)
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            if (c == 2) {
                mbar_wait(bars + 7, par);
                umma::fence_after_sync();
                umma::ld16(trow + C_X + 16 * j, zz[0]);
                umma::ld16(trow + C_X + 64 + 16 * j, zz[1]);
            }
            float (&z)[16] = zz[c & 1];
#pragma unroll
            for (int e = 0; e < 16; ++e) z[e] = tanh_mufu(z[e]);
            uint32_t pk[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) pk[e] = umma::pack_bf16(z[2 * e], z[2 * e + 1]);
            const uint4 q0 = make_uint4(pk[0], pk[1], pk[2], pk[3]), q1 = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            if (MODE == 0 && c == 0 && k > 0) mbar_wait(bars + 6, (k - 1) & 1u);      // dW1(k-1) has finished reading the ring
            *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off0) = q0;
            *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off1) = q1;
            if (MODE == 0) umma::st8_raw(trow + C_H1P + 32 * j + 8 * c, pk);         // bf16 h1 stash for P2 (this thread's own columns)
            umma::fence_proxy_async();
            umma::fence_before_sync();
            named_bar_arrive(NB_H1 + c, NB_ALL);
        }
        if (MODE == 0) umma::wait_st();

        // ================= P1: h2 = tanh(z2 + b2) in two halves, heads =================
        float h2[64];      // h2[16 cc + e] = unit 64 cc + 16 j + e
        H2_STAMP(2);
        mbar_wait(bars + 2, par);
        umma::fence_after_sync();
        H2_STAMP(3);
        {
            float z[16];
            umma::ld16(trow + C_Z2 + 16 * j, z);
#pragma unroll
            for (int e = 0; e < 16; ++e) h2[e] = z[e];
            umma::ld16(trow + C_Z2 + 64 + 16 * j, z);
#pragma unroll
            for (int e = 0; e < 16; ++e) h2[16 + e] = z[e];
        }
        umma::fence_before_sync();
        named_bar_arrive(NB_Z2A, NB_ALL);
#pragma unroll
        for (int cc = 0; cc < 2; ++cc)
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
                const float4 bb = *reinterpret_cast<const float4*>(sB2 + 64 * cc + 16 * j + 4 * e4);
                h2[16 * cc + 4 * e4 + 0] = tanh_mufu(h2[16 * cc + 4 * e4 + 0] + bb.x);
                h2[16 * cc + 4 * e4 + 1] = tanh_mufu(h2[16 * cc + 4 * e4 + 1] + bb.y);
                h2[16 * cc + 4 * e4 + 2] = tanh_mufu(h2[16 * cc + 4 * e4 + 2] + bb.z);
                h2[16 * cc + 4 * e4 + 3] = tanh_mufu(h2[16 * cc + 4 * e4 + 3] + bb.w);
            }
        H2_STAMP(4);
        mbar_wait(bars + 3, par);
        umma::fence_after_sync();
        H2_STAMP(5);
        {
            float z[16];
            umma::ld16(trow + C_Z2 + 16 * j, z);
#pragma unroll
            for (int e = 0; e < 16; ++e) h2[32 + e] = z[e];
            umma::ld16(trow + C_Z2 + 64 + 16 * j, z);
#pragma unroll
            for (int e = 0; e < 16; ++e) h2[48 + e] = z[e];
        }
        umma::fence_before_sync();
#pragma unroll
        for (int cc = 2; cc < 4; ++cc)
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
                const float4 bb = *reinterpret_cast<const float4*>(sB2 + 64 * cc + 16 * j + 4 * e4);
                h2[16 * cc + 4 * e4 + 0] = tanh_mufu(h2[16 * cc + 4 * e4 + 0] + bb.x);
                h2[16 * cc + 4 * e4 + 1] = tanh_mufu(h2[16 * cc + 4 * e4 + 1] + bb.y);
                h2[16 * cc + 4 * e4 + 2] = tanh_mufu(h2[16 * cc + 4 * e4 + 2] + bb.z);
                h2[16 * cc + 4 * e4 + 3] = tanh_mufu(h2[16 * cc + 4 * e4 + 3] + bb.w);
            }
        // head partial sums over this thread's 64 units, exchanged among the four threads of the row
        float ps[A];
#pragma unroll
        for (int a = 0; a < A; ++a) {
            ps[a] = 0.0f;
            if (a < nheads) {
                const float* w = sW4 + a * HH + 16 * j;
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
#pragma unroll
                    for (int e4 = 0; e4 < 4; ++e4) {
                        const float4 ww = *reinterpret_cast<const float4*>(w + 64 * cc + 4 * e4);
                        s0 = fmaf(h2[16 * cc + 4 * e4 + 0], ww.x, s0);
                        s1 = fmaf(h2[16 * cc + 4 * e4 + 1], ww.y, s1);
                        s2 = fmaf(h2[16 * cc + 4 * e4 + 2], ww.z, s2);
                        s3 = fmaf(h2[16 * cc + 4 * e4 + 3], ww.w, s3);
                    }
                ps[a] = (s0 + s1) + (s2 + s3);
                xch[(j * 3 + a) * TC_TILE + r] = ps[a];
            }
        }
        H2_STAMP(6);
        named_bar_sync(NB_QUAD + q, 128);
        H2_STAMP(7);
        float out[A];
#pragma unroll
        for (int a = 0; a < A; ++a) {
            out[a] = 0.0f;
            if (a < nheads)
                out[a] = ((xch[(0 * 3 + a) * TC_TILE + r] + xch[(1 * 3 + a) * TC_TILE + r]) +
                          (xch[(2 * 3 + a) * TC_TILE + r] + xch[(3 * 3 + a) * TC_TILE + r])) + sB4[net == 0 ? a : A];
        }
        if (MODE == 1) {
            const uint32_t pos = tile * TC_TILE + (uint32_t)r;
            if (j == 0 && pos < g.mb_count) {
                const size_t s = (size_t)g.mb_start + pos;
                if (net == 0) {
#pragma unroll
                    for (int a = 0; a < A; ++a) g.logits_out[s * A + a] = out[a];
                } else {
                    g.value_out[s] = out[0];
                }
            }
            named_bar_sync(NB_QUAD + q, 128);       // the exchange buffer is reused by the next tile
            continue;
        }
        mbar_wait(ring_full + b, (k >> 1) & 1u);      // long complete (the layer-1 GEMM of this tile waited for it)
        const uint4 sc = sSCAL[b * TC_TILE + r];
        const int rc_act = (int)sc.w;
        const float rc_logp_old = __uint_as_float(sc.x), rc_adv = __uint_as_float(sc.y), rc_val_old = __uint_as_float(sc.z);
        float d[A];
#pragma unroll
        for (int a = 0; a < A; ++a) d[a] = 0.0f;
        if (rc_act >= 0) {
            if (net == 0) {
                float m = out[0];
#pragma unroll
                for (int a = 1; a < A; ++a) m = fmaxf(m, out[a]);
                float se = 0.f;
#pragma unroll
                for (int a = 0; a < A; ++a) se += __expf(out[a] - m);
                const float lse = m + __logf(se);
                float lp[A], p[A];
                float ent = 0.f, new_logp = 0.f;
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    lp[a] = out[a] - lse;
                    p[a] = __expf(lp[a]);
                    ent -= p[a] * lp[a];
                    if (a == rc_act) new_logp = lp[a];
                }
                const float nadv = (rc_adv - adv_mean) * adv_rstd;
                const float logratio = new_logp - rc_logp_old;
                const float ratio = __expf(logratio);
                const float pg1 = -nadv * ratio;
                const float pg2 = -nadv * fminf(fmaxf(ratio, 1.0f - g.clip_coef), 1.0f + g.clip_coef);
                const float dpg = pg1 >= pg2 ? pg1 : 0.0f;
                if (j == 0) {
                    lsum[0] += fmaxf(pg1, pg2);
                    lsum[2] += ent;
                    lsum[3] += (ratio - 1.0f) - logratio;
                    lsum[4] += fabsf(ratio - 1.0f) > g.clip_coef ? 1.0f : 0.0f;
                }
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    const float onehot = a == rc_act ? 1.0f : 0.0f;
                    d[a] = inv_m * (dpg * (onehot - p[a]) + g.ent_coef * p[a] * (lp[a] + ent));
                    if (j == 0) gb4[a] += d[a];
                }
            } else {
                const float v = out[0];
                const float ret = rc_adv + rc_val_old;
                const float vd = v - ret;
                const float vu = vd * vd;
                const float vdiff = v - rc_val_old;
                const float vc = rc_val_old + fminf(fmaxf(vdiff, -g.clip_coef), g.clip_coef);
                const float vcd = vc - ret;
                const float vcl = vcd * vcd;
                const float gcl = (vdiff >= -g.clip_coef && vdiff <= g.clip_coef) ? vcd : 0.0f;
                const float gv = vu > vcl ? vd : (vcl > vu ? gcl : 0.5f * (vd + gcl));
                d[0] = g.vf_coef * gv * inv_m;
                if (j == 0) { lsum[1] += fmaxf(vu, vcl); gb4[0] += d[0]; }
            }
        }
        // h2 -> ring (bf16) and dout -> the free columns of the operand tile, then hand the dW4 GEMM
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            uint4 q0, q1;
            q0.x = umma::pack_bf16(h2[16 * c + 0], h2[16 * c + 1]); q0.y = umma::pack_bf16(h2[16 * c + 2], h2[16 * c + 3]);
            q0.z = umma::pack_bf16(h2[16 * c + 4], h2[16 * c + 5]); q0.w = umma::pack_bf16(h2[16 * c + 6], h2[16 * c + 7]);
            q1.x = umma::pack_bf16(h2[16 * c + 8], h2[16 * c + 9]); q1.y = umma::pack_bf16(h2[16 * c + 10], h2[16 * c + 11]);
            q1.z = umma::pack_bf16(h2[16 * c + 12], h2[16 * c + 13]); q1.w = umma::pack_bf16(h2[16 * c + 14], h2[16 * c + 15]);
            *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off0) = q0;
            *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off1) = q1;
        }
        if (j == 0) {
            __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(tOBS + b * 4096);
#pragma unroll
            for (int a = 0; a < A; ++a) {
                if (a < nheads) {
                    const int col = dout_col(O, a);
                    orow[(col >> 3) * (TC_TILE * 8) + r * 8 + (col & 7)] = __float2bfloat16_rn(d[a]);
                }
            }
        }
        umma::fence_proxy_async();
        umma::fence_before_sync();
        named_bar_arrive(NB_W4RDY, NB_ALL);
        H2_STAMP(8);
        // dz2 = (dout . W4) * (1 - h2^2), chunk by chunk: the dh1 GEMM of chunk c runs while chunk c + 1 is computed
        H2_STAMP(9);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            float dz[16];
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
                float dh[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    if (a < nheads) {
                        const float4 ww = *reinterpret_cast<const float4*>(sW4 + a * HH + 64 * c + 16 * j + 4 * e4);
                        dh[0] = fmaf(d[a], ww.x, dh[0]); dh[1] = fmaf(d[a], ww.y, dh[1]);
                        dh[2] = fmaf(d[a], ww.z, dh[2]); dh[3] = fmaf(d[a], ww.w, dh[3]);
                    }
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float hv = h2[16 * c + 4 * e4 + e];
                    dz[4 * e4 + e] = dh[e] * fmaf(-hv, hv, 1.0f);
                }
            }
            uint4 q0, q1;
            q0.x = umma::pack_bf16(dz[0], dz[1]); q0.y = umma::pack_bf16(dz[2], dz[3]); q0.z = umma::pack_bf16(dz[4], dz[5]); q0.w = umma::pack_bf16(dz[6], dz[7]);
            q1.x = umma::pack_bf16(dz[8], dz[9]); q1.y = umma::pack_bf16(dz[10], dz[11]); q1.z = umma::pack_bf16(dz[12], dz[13]); q1.w = umma::pack_bf16(dz[14], dz[15]);
            if (c == 0) {
                mbar_wait(bars + 4, par);          // the dW4 GEMM has consumed the h2 chunks
                H2_STAMP(10);
            }
            *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off0) = q0;
            *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off1) = q1;
            umma::fence_proxy_async();
            umma::fence_before_sync();
            named_bar_arrive(NB_DZ2 + c, NB_ALL);
        }

        // ================= P2: dz1 = dh1 * (1 - h1^2) =================
        uint32_t hq[NCH][8];   // this thread's h1 values (bf16 pairs) back from their tensor-memory stash
#pragma unroll
        for (int c = 0; c < NCH; ++c) umma::ld8_raw(trow + C_H1P + 32 * j + 8 * c, hq[c]);
        H2_STAMP(11);
        mbar_wait(bars + 5, par);          // dh1 complete (and the ring's dz2 chunks staged)
        umma::fence_after_sync();
        H2_STAMP(12);
        {
            float dhu[2][16];          // chunks 2, 3 first: their columns are where layer 1 of the next tile goes
            umma::ld16(trow + C_DH + 64 * 2 + 16 * j, dhu[0]);
            umma::ld16(trow + C_DH + 64 * 3 + 16 * j, dhu[1]);
            umma::fence_before_sync();
            if (k + 1 < nmy) named_bar_arrive(NB_Z2A, NB_ALL);
#pragma unroll
            for (int cc = 0; cc < NCH; ++cc) {
                const int c = (cc + 2) & 3;
                float dh[16];
                if (cc < 2) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) dh[e] = dhu[cc][e];
                } else {
                    umma::ld16(trow + C_DH + 64 * c + 16 * j, dh);
                }
                uint4 o4[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t* qv = hq[c] + 4 * h;
                    const float hv[8] = {umma::bf16_lo(qv[0]), umma::bf16_hi(qv[0]), umma::bf16_lo(qv[1]), umma::bf16_hi(qv[1]),
                                         umma::bf16_lo(qv[2]), umma::bf16_hi(qv[2]), umma::bf16_lo(qv[3]), umma::bf16_hi(qv[3])};
                    float z[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) z[e] = dh[8 * h + e] * fmaf(-hv[e], hv[e], 1.0f);
                    o4[h].x = umma::pack_bf16(z[0], z[1]); o4[h].y = umma::pack_bf16(z[2], z[3]);
                    o4[h].z = umma::pack_bf16(z[4], z[5]); o4[h].w = umma::pack_bf16(z[6], z[7]);
                }
                *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off0) = o4[0];
                *reinterpret_cast<uint4*>(tACT + c * SLOT_BYTES + off1) = o4[1];
            }
        }
        umma::fence_proxy_async();
        umma::fence_before_sync();
        named_bar_arrive(NB_DZ1, NB_ALL);
        H2_STAMP(13);
    }

    if (MODE == 1) {
        umma::fence_before_sync();
        __syncthreads();
        if (warp == 1) umma::tmem_dealloc(tmem, TM_COLS);
        return;
    }

    // ================= epilogue: add this CTA's small partial gradients to its row =================
    mbar_wait(bars + 6, (nmy - 1) & 1u);       // the last commit: every GEMM of this CTA has completed
    umma::fence_after_sync();
    float* part = g.grad_part + (size_t)blockIdx.x * g.ppad;
    const int base = net * P::C_ACTOR;
    const int nout = net == 0 ? A : 1;
    const float keep = g.first ? 0.0f : 1.0f;      // first launch of the minibatch: overwrite the row (it holds the previous minibatch)
    auto accum = [&](int i, float v) { part[i] = g.first ? v : part[i] + v; };
    if (warp < 4) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int o = 128 * u + r;
            float v16[16];
            umma::ld16(trow + C_SW1 + 16 * u, v16);
#pragma unroll
            for (int i = 0; i < O; ++i) accum(base + o * O + i, v16[i] + v16[8 + i]);           // dW1 = dz1^T . (obs_hi + obs_lo)
            accum(base + HH * O + o, v16[O]);                                                   // db1
            umma::ld16(trow + C_SW4 + 16 * u, v16);
#pragma unroll
            for (int a = 0; a < A; ++a)
                if (a < nout) accum(base + P::C_NET + a * HH + o, v16[dout_col(O, a)]);          // dW4
        }
    }
    {
        float vals[8] = {lsum[0], lsum[1], lsum[2], lsum[3], lsum[4], gb4[0], gb4[1], gb4[2]};
#pragma unroll
        for (int x = 0; x < 8; ++x) {
            const float sv = warp_sum(vals[x]);
            if (lane == 0) red[warp * 12 + x] = sv;
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 8) {
        float sv = 0.0f;
#pragma unroll
        for (int w = 0; w < TC_COMPUTE / 32; ++w) sv += red[w * 12 + tid];
        if (tid < 5) g.loss_part[blockIdx.x * LOSS_TERMS + tid] = keep * g.loss_part[blockIdx.x * LOSS_TERMS + tid] + sv;
        else if (tid - 5 < nout) accum(base + P::C_NET + nout * HH + (tid - 5), sv);            // head biases
    }
    if (warp == 1) umma::tmem_dealloc(tmem, TM_COLS);
}

// ---------------------------------------------------------------------------------------------------------------------
// dW2 = dz2^T . h1 over the staged tiles of one launch of mlp256_kernel: split-K, one net per CTA.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int B_STAGES = 3;
constexpr int B_STAGE_BYTES = 65536;      // 64 samples: dz2 [4 chunks][64 rows][128 B] + h1 the same
constexpr int B_BLOCK = 192;              // producer warp, issuer warp, four epilogue warps

__global__ void __launch_bounds__(B_BLOCK, 1) dw2_gemm256_kernel(const unsigned char* __restrict__ stage_dz,
                                                                 const unsigned char* __restrict__ stage_h1, uint32_t stage_tiles,
                                                                 uint32_t ntiles, float* __restrict__ grad_part, int ppad, int c_actor,
                                                                 int w2_off, int first) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + B_STAGES * B_STAGE_BYTES);     // full[3], empty[3], done
    uint32_t* slot = reinterpret_cast<uint32_t*>(bars + 2 * B_STAGES + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int net = blockIdx.x & 1;
    const uint32_t cin = blockIdx.x >> 1, ncn = gridDim.x >> 1;
    if (cin >= ntiles) return;
    const uint32_t nmy = (ntiles - cin + ncn - 1) / ncn;
    const uint32_t nit = 2 * nmy;             // half-tiles of 64 samples

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < B_STAGES; ++i) { mbar_init(bars + i, 1); mbar_init(bars + B_STAGES + i, 1 + 4); }   // empty: MMA commit + 4 warps
        mbar_init(bars + 2 * B_STAGES, 1);
        mbar_fence_init();
    }
    if (warp == 2) umma::tmem_alloc(slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *slot;

    if (warp == 0) {
        if (lane == 0) {
            for (uint32_t it = 0; it < nit; ++it) {
                const uint32_t s = it % B_STAGES, use = it / B_STAGES;
                if (it >= (uint32_t)B_STAGES) mbar_wait(bars + B_STAGES + s, (use - 1u) & 1u);
                const uint32_t tile = cin + (it >> 1) * ncn, half = it & 1u;
                const unsigned char* src_dz = stage_dz + ((size_t)net * stage_tiles + tile) * TILE_BYTES + half * 8192;
                const unsigned char* src_h1 = stage_h1 + ((size_t)net * stage_tiles + tile) * TILE_BYTES + half * 8192;
                unsigned char* dst = sm + s * B_STAGE_BYTES;
                mbar_expect_tx(bars + s, (uint32_t)B_STAGE_BYTES);
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    bulk_g2s(dst + c * 8192, src_dz + c * SLOT_BYTES, 8192u, bars + s);
                    bulk_g2s(dst + 32768 + c * 8192, src_h1 + c * SLOT_BYTES, 8192u, bars + s);
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t ID_W2 = umma::make_idesc(128, 256, true, true);
        for (uint32_t it = 0; it < nit; ++it) {
            const uint32_t s = it % B_STAGES, use = it / B_STAGES;
            mbar_wait(bars + s, use & 1u);
            umma::fence_after_sync();
            if (umma::elect_one()) {
                const uint32_t adz = smem_u32(sm + s * B_STAGE_BYTES), ah1 = adz + 32768;
#pragma unroll
                for (int kb = 0; kb < 4; ++kb)
#pragma unroll
                    for (int u = 0; u < 2; ++u)
                        umma::mma(tmem + 256 * u, umma::make_desc(adz + u * 16384 + kb * 2048, 8192, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(ah1 + kb * 2048, 8192, 1024, umma::LAYOUT_SW128), ID_W2, (it > 0 || kb > 0) ? 1u : 0u);
                umma::commit(bars + B_STAGES + s);
                if (it == nit - 1) umma::commit(bars + 2 * B_STAGES);
            }
            __syncwarp();
        }
    } else {
        // warps 2..5.  During the main loop: db2 = column sums of dz2 -- warp w owns chunk w - 2 (64 units), lane l the unit pair
        // (2l, 2l + 1) = one 32-bit word of every row of the chunk's SW128 image.
        const int cw = warp - 2;
        float sb0 = 0.0f, sb1 = 0.0f;
        for (uint32_t it = 0; it < nit; ++it) {
            const uint32_t s = it % B_STAGES, use = it / B_STAGES;
            mbar_wait(bars + s, use & 1u);
            const unsigned char* ch = sm + s * B_STAGE_BYTES + cw * 8192;
#pragma unroll 8
            for (int rr = 0; rr < 64; ++rr) {
                const uint32_t w = *reinterpret_cast<const uint32_t*>(ch + rr * 128 + ((((lane >> 2) ^ (rr & 7))) << 4) + (lane & 3) * 4);
                sb0 += umma::bf16_lo(w);
                sb1 += umma::bf16_hi(w);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + B_STAGES + s);
        }
        {
            float* pb2 = grad_part + (size_t)blockIdx.x * ppad + net * c_actor + w2_off + HH * HH + 64 * cw + 2 * lane;
            pb2[0] = first ? sb0 : pb2[0] + sb0;
            pb2[1] = first ? sb1 : pb2[1] + sb1;
        }
        // epilogue: TMEM lane quadrant = warp % 4
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
        mbar_wait(bars + 2 * B_STAGES, 0);
        umma::fence_after_sync();
        named_bar_sync(1, 128);      // all four warps are done reading the stage ring (db2 sums) before any of them reuses it below
        // The accumulator row of a thread is one row of dW2 (1 KB): written straight from registers, a warp would touch 32
        // different lines per instruction.  Each 32 x 32 block goes through shared memory instead (the stage ring is idle now)
        // and leaves as 32 coalesced 128-byte rows.
        float* part = grad_part + (size_t)blockIdx.x * ppad + net * c_actor + w2_off;
        float* tile = reinterpret_cast<float*>(sm) + (warp - 2) * (32 * 33);
#pragma unroll 1
        for (int u = 0; u < 2; ++u) {
#pragma unroll 1
            for (int cb = 0; cb < 8; ++cb) {
                float v[32];
                umma::ld32(trow + 256 * u + 32 * cb, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) tile[lane * 33 + i] = v[i];
                __syncwarp();
                float* dst = part + (size_t)(128 * u + 32 * q) * HH + 32 * cb + lane;
#pragma unroll 8
                for (int rr = 0; rr < 32; ++rr) {
                    const float x = tile[rr * 33 + lane];
                    dst[(size_t)rr * HH] = first ? x : dst[(size_t)rr * HH] + x;
                }
                __syncwarp();
            }
        }
        umma::fence_before_sync();
    }
    __syncthreads();
    if (warp == 2) umma::tmem_dealloc(tmem, 512);
}

template <int O, int A, int OP, int RW>
static int launch_grad256_t(const GradArgs& g0, int P, float* grad_out, float* loss_terms_out, void* workspace, cudaStream_t st) {
    const WorkspaceLayout w = workspace_layout(P, HH);
    int grid = sm_count();
    if (grid > MAX_GRAD_CTAS) grid = MAX_GRAD_CTAS;
    grid &= ~1;
    const int smem_a = Smem256<O, A>::TOTAL;
    const int smem_b = B_STAGES * B_STAGE_BYTES + 128 + 1024;
    DRL_CUDA(cudaFuncSetAttribute(mlp256_kernel<O, A, OP, RW, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_a));
    DRL_CUDA(cudaFuncSetAttribute(dw2_gemm256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_b));
    Grad256Args a;
    a.packed = g0.packed; a.rec = g0.rec; a.idx = g0.idx; a.mb_total = g0.mb_count; a.adv_stats = g0.adv_stats;
    a.clip_coef = g0.clip_coef; a.ent_coef = g0.ent_coef; a.vf_coef = g0.vf_coef;
    a.stage_h1 = reinterpret_cast<unsigned char*>(workspace) + w.stage;
    a.stage_dz = a.stage_h1 + (size_t)2 * STAGE_TILES * TILE_BYTES;
    a.stage_tiles = STAGE_TILES;
    a.grad_part = g0.grad_part; a.loss_part = g0.loss_part; a.ppad = g0.ppad;
    a.logits_out = nullptr; a.value_out = nullptr; a.only_net = -1; a.dbg = g0.dbg;
    const uint32_t chunk = (uint32_t)STAGE_TILES * TC_TILE;
    for (uint32_t off = 0; off < g0.mb_count; off += chunk) {
        a.mb_start = g0.mb_start + off;
        a.mb_count = g0.mb_count - off < chunk ? g0.mb_count - off : chunk;
        const uint32_t ntiles = (a.mb_count + TC_TILE - 1) / TC_TILE;
        a.first = off == 0 ? 1 : 0;
        mlp256_kernel<O, A, OP, RW, 0><<<grid, A_BLOCK, smem_a, st>>>(a);
        DRL_LAUNCH_CHECK("mlp256_kernel");
        dw2_gemm256_kernel<<<grid, B_BLOCK, smem_b, st>>>(a.stage_dz, a.stage_h1, a.stage_tiles, ntiles, a.grad_part, a.ppad,
                                                        Packed256<O, A>::C_ACTOR, Packed256<O, A>::W2_OFF, a.first);
        DRL_LAUNCH_CHECK("dw2_gemm256_kernel");
    }
    // rows that took part: CTA c works iff (c >> 1) < tiles of the (largest = first) chunk; even rows hold actor entries, odd
    // rows critic entries, so each parameter is folded over the rows of its own net only
    const uint32_t first_tiles = ((g0.mb_count < chunk ? g0.mb_count : chunk) + TC_TILE - 1) / TC_TILE;
    const int active = (int)(2 * first_tiles < (uint32_t)grid ? 2 * first_tiles : (uint32_t)grid);
    return launch_grad_reduce(g0, active, P, 2, Packed256<O, A>::C_ACTOR, grad_out, loss_terms_out, st);
}

int launch_grad256(const drl_net_t* net, const GradArgs& g, int P, float* grad_out, float* loss_terms_out, void* workspace,
                   cudaStream_t st) {
    if (net->obs_dim == 4) return launch_grad256_t<4, 2, 4, 8>(g, P, grad_out, loss_terms_out, workspace, st);
    if (net->obs_dim == 2) return launch_grad256_t<2, 3, 4, 8>(g, P, grad_out, loss_terms_out, workspace, st);
    return launch_grad256_t<6, 3, 8, 16>(g, P, grad_out, loss_terms_out, workspace, st);
}

template <int O, int A, int OP>
static int launch_forward256_t(const float* packed, const float* obs, int64_t n, float* logits, float* value, int only_net, cudaStream_t st) {
    int grid = sm_count();
    if (grid > MAX_GRAD_CTAS) grid = MAX_GRAD_CTAS;
    grid &= ~1;
    const int smem_a = Smem256<O, A>::TOTAL;
    DRL_CUDA(cudaFuncSetAttribute(mlp256_kernel<O, A, OP, 8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_a));
    Grad256Args a;
    memset(&a, 0, sizeof(a));
    a.packed = packed; a.rec = obs; a.logits_out = logits; a.value_out = value; a.only_net = only_net;
    const int64_t chunk = (int64_t)1 << 30;
    for (int64_t off = 0; off < n; off += chunk) {
        a.mb_start = (uint32_t)off; a.mb_count = (uint32_t)(n - off < chunk ? n - off : chunk); a.mb_total = a.mb_count;
        mlp256_kernel<O, A, OP, 8, 1><<<grid, A_BLOCK, smem_a, st>>>(a);
        DRL_LAUNCH_CHECK("mlp256_kernel (forward)");
    }
    return DRL_OK;
}

// only_net: -1 = both nets (logits and values), 0 = actor only, 1 = critic only (the value pass after the 256-wide rollout)
int launch_forward256(const drl_net_t* net, const float* packed, const float* obs, int64_t n, float* logits, float* value,
                      int only_net, cudaStream_t st) {
    if (net->obs_dim == 4) return launch_forward256_t<4, 2, 4>(packed, obs, n, logits, value, only_net, st);
    if (net->obs_dim == 2) return launch_forward256_t<2, 3, 4>(packed, obs, n, logits, value, only_net, st);
    return launch_forward256_t<6, 3, 8>(packed, obs, n, logits, value, only_net, st);
}

}  // namespace h256
}  // namespace drl
