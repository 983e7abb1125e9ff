// update_tc.cu -- tensor-core (tcgen05 / TMEM) implementation of the PPO minibatch gradient,
// deep_rl/ppo.py:159-190.  Same inputs, outputs and per-CTA partial-gradient format as ppo_grad_kernel
// (update_ops.cu); operands of the GEMMs are bf16, accumulation is fp32 in tensor memory.
//
// One persistent CTA per SM: 16 compute warps + 1 MMA-issuer warp + 1 loader warp.  A tile is 128 samples = the 128 TMEM lanes;
// compute thread (warp w, lane l) owns sample row r = 32*(w&3)+l, net (w>>3) (0 = actor trunk, 1 = critic trunk) and
// hidden units [32*((w>>2)&1), +32) of that net, i.e. four threads share a row.  Work per tile k:
//   MMA    l1(k):   z1 = [obs_hi|1|obs_lo] . [W1|b1|W1]^T (per net M128 N64 K16, no swizzle; the operand tile comes from the loader)
//   P0(k)  tcgen05.ld z1, tanh, h1 -> bf16 SW128 tile
//   MMA    fwd(k):  z2 = h1 . W2^T                      (per net M128 N64 K64, A/B K-major)
//   P1(k)  tcgen05.ld z2, tanh, heads, clipped-surrogate / value / entropy loss and their closed-form output
//          gradients, dz2 = (dout . W4) * (1 - h2^2); h2, dz2, dout -> bf16 tiles
//   MMA    dh1(k):  dh1 = dz2 . W2                      (M128 N64 K64, B MN-major: the same W2 tile, transposed by descriptor)
//   MMA    wg(k):   dW4 += h2^T . dout   db2 += dz2^T . [obs|1]          (M128 N16 K128)
//                   dW2 += dz2^T . h1                   (M128 N128 K128, both operands MN-major: the activation tiles again)
//                   -- issued AFTER fwd(k+1): nobody waits for them until late in X(k+1)
//   P2(k)  tcgen05.ld dh1, dz1 = dh1 * (1 - h1^2) -> bf16 tile
//   MMA    w1(k):   [dW1|db1] += dz1^T . [obs|1]        (M128 N16 K128)
// The loop is software-pipelined and warp-specialised so that no compute warp waits for a GEMM it has just
// handed over, and no CTA-wide barrier sits in the loop:
//   X(k): wait fwd(k), P1(k), hand dh1(k)   Y(k): wait l1(k+1), P0(k+1), hand fwd(k+1)   Z(k): wait dh1(k), P2(k), hand w1(k)
// "hand" = fence.proxy.async + bar.arrive on a named barrier; the issuer warp bar.syncs on it, issues the
// tcgen05.mma group and commits to an mbarrier the compute warps wait on.  h1 tiles are double-buffered, z2 and dh1
// have separate TMEM columns.  The gather is decoupled from the compute warps: the loader warp reads the permuted
// indices and the 32/64-byte records of tile k+2 (plain global loads; their latency and their scoreboards stay in that
// warp), writes the [obs_hi|1|obs_lo] operand tile and the per-row scalars {logp, adv, val, act} into a three-deep
// shared-memory ring and signals a "full" mbarrier; the slot is handed back by a tcgen05.commit after the last GEMM that
// reads it.  All weight-gradient accumulators live in TMEM for the whole kernel (432 of 512 columns used) and are
// written once, as this CTA's partial gradient, at the end.
#include "drl_pack.cuh"
#include "drl_tc_common.cuh"
#include "drl_update.cuh"

namespace drl {

// TMEM columns
constexpr uint32_t C_ZF = 0, C_DH = 128, C_W2 = 256, C_B2 = 384, C_W4 = 400, C_W1 = 416, TC_COLS = 512;

template <int O, int A>
struct TcSmem {
    using P = Packed<O, A>;
    static constexpr int W_BYTES = (P::TC_END - P::TC_W2) * 4;   // bf16 W2 tiles (16 KB) + fp32 small weights
    static constexpr int OFF_W = 0;
    static constexpr int OFF_H1 = (OFF_W + W_BYTES + 1023) / 1024 * 1024;   // two buffers x (actor, critic) x 16 KB
    static constexpr int OFF_H2 = OFF_H1 + 65536;
    static constexpr int OFF_DZ = OFF_H2 + 32768;
    static constexpr int OFF_DZ1 = OFF_DZ + 32768;     // dz1 has its own tile: the dz2 readers (dW2, db2) may still be running
    static constexpr int OFF_OBS = OFF_DZ1 + 32768;    // three NS16 buffers [obs_hi|1|obs_lo] (tile % 3)
    static constexpr int OFF_DOUT = OFF_OBS + 12288;   // one NS16 buffer
    static constexpr int OFF_SCAL = OFF_DOUT + 4096;   // three buffers of per-row scalars {logp_old, adv, val_old, act} (16 B each)
    static constexpr int OFF_BAR = OFF_SCAL + 3 * 2048;   // 13 mbarriers + TMEM slot
    static constexpr int OFF_XCH = OFF_BAR + 128;      // head partial sums [net][half][A][128 rows] fp32
    static constexpr int OFF_RED = OFF_XCH + 2 * 2 * 4 * 128 * 4;
    static constexpr int OFF_CTX = OFF_RED + 16 * 12 * 4;        // TailCtx: the tail's arguments, copied from the kernel parameters once
    static constexpr int TOTAL = OFF_CTX + 512 + 1024;           // + alignment slack
    static_assert(TOTAL <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
};

// diagnostics, only in a -DDRL_TC_STAMPS build (profiles/tc_stamps.py): cycle stamps of CTA 0 (slot = tile * 16 + event) and
// whole-kernel stamps of CTA 0 / thread 0 (slots 8..15 of the issuer rows of the debug block)
#ifdef DRL_TC_STAMPS
#define TC_STAMP(ev) do { if (g.dbg != nullptr && blockIdx.x == 0 && lane == 0 && k < 12 && (warp == 0 || warp == TC_COMPUTE / 32)) g.dbg[(warp == 0 ? 0 : 256) + k * 16 + (ev)] = clock64(); } while (0)
#define TC_KSTAMP(n) do { if (g.dbg != nullptr && blockIdx.x == 0 && tid == 0) g.dbg[256 + ((n) >> 3) * 16 + 8 + ((n) & 7)] = clock64(); } while (0)
#else
#define TC_STAMP(ev) do { } while (0)
#define TC_KSTAMP(n) do { } while (0)
#endif

enum : uint32_t { BAR_FWD = 1, BAR_BWD = 2, BAR_W1 = 3, BAR_PAIR0 = 4, BAR_L1 = 12 };   // named barriers (0 = __syncthreads)

constexpr int GRAD_TC_BLOCK = TC_THREADS + 32;   // + the loader warp
constexpr int RING = 3;                          // depth of the [obs|1] / scalar ring

// sample id of row r of this CTA's tile `tile` (0xFFFFFFFF = padding row)
__device__ __forceinline__ uint32_t tc_sample_index(const GradArgs& g, uint32_t mb_start, uint32_t mb_count, uint32_t tile, uint32_t ntiles, int r) {
    const uint32_t pos = tile * TC_TILE + (uint32_t)r;
    if (tile >= ntiles || pos >= mb_count) return 0xFFFFFFFFu;
    const uint32_t i = mb_start + pos;
    return g.idx ? __ldg(g.idx + i) : i;
}

// What the tail reads of the kernel parameters.  The tail is a separate function, and a reference to the parameter block would
// turn every field access into a generic load; thread 0 copies the block into shared memory once per launch instead.
struct TailCtx {
    TailArgs tl;
    float* grad_part; float* loss_part; float* packed; long long* dbg;
    int ppad; uint32_t mb_count; float ent_coef, vf_coef;
};
static_assert(sizeof(TailCtx) <= 512, "TailCtx block");

// ================= in-kernel tail of one minibatch: fold partials, [all-reduce over NVLink peer memory], clip, Adam, reload =================
// Only the 512 compute threads take part: named barrier 13, count 512.  A separate (not inlined) function: its registers (20
// loads in flight in the fold, the Adam state) are then allocated apart from the tile loop's, which otherwise spills.
template <int O, int A>
__device__ __noinline__ void tc_tail_step(const TailCtx* cx, uint32_t s, uint32_t nsteps, unsigned char* sm, uint64_t* bars) {
    using P = Packed<O, A>;
    using S = TcSmem<O, A>;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const struct { long long* dbg; } g = {cx->dbg};      // for the stamp macros
    (void)g;
    // ================= in-kernel tail: fold partials, [all-reduce over NVLink peer memory], clip, Adam =================
    // Only the 512 compute threads take part: named barrier 13, count 512.
    constexpr uint32_t BAR_TAIL = 13;
    const TailArgs& tl = cx->tl;
    const AdamArgs& ad = tl.a;
    const int PP = ad.P;
    float neg_step_size = tl.neg_step_size_s[s], bc2_sqrt = tl.bc2_sqrt_s[s];
    uint32_t seq = tl.seq + s;
    if (tl.ctrl != nullptr) {        // counters of a graph-replayed update live in device memory
        neg_step_size = tl.ctrl->neg_step_size[tl.ordinal + s];
        bc2_sqrt = tl.ctrl->bc2_sqrt[tl.ordinal + s];
        seq = tl.ctrl->comm_seq + (uint32_t)(tl.ordinal + s) + 1u;
    }
    float* const loss_terms_out = tl.loss_terms_out != nullptr ? tl.loss_terms_out + LOSS_TERMS * s : nullptr;
    const uint32_t bar_target = (s + 1u) * gridDim.x;      // the grid-barrier counters count on through the minibatches of the launch
    const int nparts = gridDim.x;
    float* tred = reinterpret_cast<float*>(sm + S::OFF_H1);              // [8][64] fold scratch (tiles are dead now)
    double* dred = reinterpret_cast<double*>(sm + S::OFF_H1 + 4096);     // [16] warp partials of the squared norm
    float* sbc = reinterpret_cast<float*>(sm + S::OFF_H1 + 8192);        // broadcast slot
    // All CTAs are co-resident (cooperative launch).  The CTA's writes are ordered before thread 0's release-increment by the
    // named barrier (the release is cumulative), the acquire-load orders the other CTAs' writes before everything after the
    // second named barrier: one thread fences, once per side, instead of a sequentially-consistent fence in all 512.
    auto grid_barrier = [&](uint32_t* ctr) {
        named_bar_sync(BAR_TAIL, TC_COMPUTE);
        if (tid == 0) {
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
            uint32_t seen;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(ctr) : "memory");
            } while (seen < bar_target);
        }
        named_bar_sync(BAR_TAIL, TC_COMPUTE);
    };
    grid_barrier(tl.ctr + 0);                     // every CTA's partial gradient is in global memory
    TC_KSTAMP(6);
    const int chunk = (PP + nparts - 1) / nparts;
    const int p_lo = blockIdx.x * chunk, p_hi = min(PP, p_lo + chunk);
    const int pl = tid & 63, sl = tid >> 6;        // parameter within a group of 64, slice of the partials (8 slices)
    const bool multi = tl.world > 1;
    const CommLayout cl = comm_layout(PP);
    const uint32_t gen = seq & 1u;
    double sq = 0.0;
    for (int p0 = p_lo; p0 < p_hi; p0 += 64) {
        const int p = p0 + pl;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        if (p < p_hi) {
            // all (up to 20) loads of this thread in flight at once: one L2 round trip instead of seven.  The summation
            // keeps the association of grad_reduce_kernel: four interleaved accumulators over groups of 32 partials while a
            // whole group fits, then the remaining partials one by one into the first accumulator.
            static_assert(MAX_GRAD_CTAS <= 160, "fold is unrolled for at most 160 partials");
            float pv[20];
#pragma unroll
            for (int j = 0; j < 20; ++j) {
                const int c = sl + 8 * j;
                pv[j] = c < nparts ? __ldcg(cx->grad_part + (size_t)c * cx->ppad + p) : 0.0f;
            }
            bool rest = false;
#pragma unroll
            for (int gq = 0; gq < 5; ++gq) {
                const int c = sl + 32 * gq;
                if (!rest && c + 24 < nparts) {
                    a0 += pv[4 * gq]; a1 += pv[4 * gq + 1]; a2 += pv[4 * gq + 2]; a3 += pv[4 * gq + 3];
                } else {
                    rest = true;
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (c + 8 * q < nparts) a0 += pv[4 * gq + q];
                }
            }
        }
        tred[sl * 64 + pl] = (a0 + a1) + (a2 + a3);
        named_bar_sync(BAR_TAIL, TC_COMPUTE);
        if (sl == 0 && p < p_hi) {
            float t = tred[pl];
#pragma unroll
            for (int y = 1; y < 8; ++y) t += tred[y * 64 + pl];
            if (multi) {
                // push: this rank's folded value goes into slot `rank` of EVERY rank's symmetric buffer (remote stores over NVLink
                // are posted; nobody has to fetch it later)
                for (int rk = 0; rk < tl.world; ++rk)
                    reinterpret_cast<float*>(tl.peer[rk] + cl.xgrad[gen] + (size_t)tl.rank * cl.rank_stride)[p] = t;
            } else {
                tl.grad_out[p] = t;
                const double gs = (double)(t * ad.grad_scale);
                sq = fma(gs, gs, sq);
            }
        }
        named_bar_sync(BAR_TAIL, TC_COMPUTE);
    }
    TC_KSTAMP(7);
    if (multi) {
        // ---- one-shot all-reduce over NVLink, slice by slice: every CTA publishes ITS slice with its own flag in every peer's
        // buffer as soon as the slice is folded, and waits only for the same slice of the other ranks (no grid-wide barrier) ----
        if (sl == 0) __threadfence_system();          // the threads that wrote: their remote stores are ordered before the flag
        named_bar_sync(BAR_TAIL, TC_COMPUTE);
        if (tid < tl.world) {
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t*>(tl.peer[tid] + cl.flags[gen] + sizeof(uint32_t) * (tl.rank * FLAG_CTAS + blockIdx.x)) = seq;
            const volatile uint32_t* f = reinterpret_cast<const volatile uint32_t*>(tl.peer[tl.rank] + cl.flags[gen] +
                                                                                    sizeof(uint32_t) * (tid * FLAG_CTAS + blockIdx.x));
            const long long t0 = clock64();
            while (*f < seq) {
                if (clock64() - t0 > 40000000000ll) {   // ~20 s: a peer is gone (start-up skew between ranks can reach seconds)
                    if (tl.error_flag) { *reinterpret_cast<volatile int*>(tl.error_flag) = 1; __threadfence(); }
                    break;
                }
            }
            __threadfence_system();
        }
        named_bar_sync(BAR_TAIL, TC_COMPUTE);
        const float* mine = reinterpret_cast<const float*>(tl.peer[tl.rank] + cl.xgrad[gen]);
        for (int p = p_lo + tid; p < p_hi; p += TC_COMPUTE) {
            float t = 0.0f;
            for (int rk = 0; rk < tl.world; ++rk)                      // rank order: the same sum on every rank
                t += __ldcg(mine + (size_t)rk * (cl.rank_stride / sizeof(float)) + p);
            tl.grad_out[p] = t;
            const double gs = (double)(t * ad.grad_scale);
            sq = fma(gs, gs, sq);
        }
    }
    sq = warp_sum(sq);
    if (lane == 0) dred[warp] = sq;
    named_bar_sync(BAR_TAIL, TC_COMPUTE);
    if (tid == 0) {
        double t = 0.0;
        for (int wv = 0; wv < TC_COMPUTE / 32; ++wv) t += dred[wv];
        tl.cta_sumsq[blockIdx.x] = t;
    }
    TC_KSTAMP(8);
    // optimizer state of this thread's first parameter: fetched before the barrier, it does not depend on the norm
    const int p_first = p_lo + tid;
    float pre_m = 0.f, pre_v = 0.f, pre_w = 0.f;
    if (p_first < p_hi) { pre_m = ad.m[p_first]; pre_v = ad.v[p_first]; pre_w = ad.params[p_first]; }
    grid_barrier(tl.ctr + 2);                     // every CTA's squared-norm share is published
    TC_KSTAMP(9);
    if (warp == 0) {
        double tot = 0.0;
        for (int i = lane; i < nparts; i += 32) tot += __ldcg(tl.cta_sumsq + i);
        tot = warp_sum(tot);
        if (lane == 0) sbc[0] = clip_coef(tot, ad);
    } else if (blockIdx.x == 0 && warp >= 1 && warp <= 5 && loss_terms_out != nullptr) {
        float t = 0.f;                                    // warp w folds loss term w-1 over the CTAs
        for (int c = lane; c < nparts; c += 32) t += __ldcg(cx->loss_part + c * LOSS_TERMS + (warp - 1));
        t = warp_sum(t);
        if (lane == 0) sbc[4 + warp - 1] = t;
    }
    named_bar_sync(BAR_TAIL, TC_COMPUTE);
    const float coef = sbc[0];
    // A peer that missed the all-reduce timeout left garbage in the summed gradient: skip the optimizer step on every CTA
    // (the flag was written before the grid barrier above, so all CTAs agree; it is sticky, the host raises on its next read).
    const bool peer_lost = multi && tl.error_flag != nullptr && *reinterpret_cast<volatile int*>(tl.error_flag) != 0;
    for (int p = p_lo + tid; p < p_hi && !peer_lost; p += TC_COMPUTE) {
        const float gsc = (__ldcg(tl.grad_out + p) * ad.grad_scale) * coef;
        float m, v, wgt;
        if (p == p_first) { m = pre_m; v = pre_v; wgt = pre_w; }
        else { m = ad.m[p]; v = ad.v[p]; wgt = ad.params[p]; }
        adam_apply(gsc, m, v, wgt, ad.om_beta1, ad.beta2, ad.om_beta2, ad.eps, neg_step_size, bc2_sqrt);
        ad.m[p] = m; ad.v[p] = v; ad.params[p] = wgt;
        if (ad.packed != nullptr) packed_store<O, A>(ad.packed, p, wgt);
    }
    TC_KSTAMP(10);
    if (blockIdx.x == 0 && tid == 0 && loss_terms_out != nullptr)
        store_loss_terms(loss_terms_out, sbc + 4, cx->mb_count, cx->ent_coef, cx->vf_coef);
    if (s + 1 < nsteps) {
        // next minibatch of the launch: every CTA has applied its slice of the Adam step (and refreshed its part of the packed
        // weights) -> reload the weight tiles; the loader has the first [obs|1] tiles in the ring already
        grid_barrier(tl.ctr + 1);
        if (tid == 0) {
            asm volatile("fence.proxy.async;" ::: "memory");      // other CTAs' generic-proxy stores -> this thread's TMA reads
            mbar_expect_tx(bars, (uint32_t)S::W_BYTES);
            const char* src = reinterpret_cast<const char*>(cx->packed + P::TC_W2);
            for (uint32_t off = 0; off < (uint32_t)S::W_BYTES; off += 16384u) {
                const uint32_t nb = (uint32_t)S::W_BYTES - off < 16384u ? (uint32_t)S::W_BYTES - off : 16384u;
                bulk_g2s(sm + S::OFF_W + off, src + off, nb, bars);
            }
        }
    } else if (tid == 0) {
        __threadfence();
        if (atomicAdd(tl.ctr + 3, 1u) == gridDim.x - 1) { tl.ctr[0] = 0u; tl.ctr[1] = 0u; tl.ctr[2] = 0u; tl.ctr[3] = 0u; }   // re-arm
    }
}

template <int O, int A, int OP, int RW>
__global__ void __launch_bounds__(GRAD_TC_BLOCK, 1) ppo_grad_tc_kernel(const __grid_constant__ GradArgs g) {
    using P = Packed<O, A>;
    using S = TcSmem<O, A>;
    constexpr int OW = P::OW;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* tW2 = sm + S::OFF_W;
    const float* sW1 = reinterpret_cast<const float*>(sm + S::OFF_W + 2 * H * H * 2);
    const float* sB1 = sW1 + 2 * H * OW;
    const float* sB2 = sB1 + 2 * H;
    const float* sW4 = sB2 + 2 * H;
    const float* sB4 = sW4 + (A + 1) * H;
    unsigned char* tW1B = reinterpret_cast<unsigned char*>(const_cast<float*>(sB4 + 4));   // bf16 layer-1 B tiles
    unsigned char* tH1 = sm + S::OFF_H1;
    unsigned char* tH2 = sm + S::OFF_H2;
    unsigned char* tDZ = sm + S::OFF_DZ;
    unsigned char* tDZ1 = sm + S::OFF_DZ1;
    unsigned char* tOBS = sm + S::OFF_OBS;
    unsigned char* tDOUT = sm + S::OFF_DOUT;
    uint4* sSCAL = reinterpret_cast<uint4*>(sm + S::OFF_SCAL);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + S::OFF_BAR);   // 0 weights, 1 fwd, 2 dh1, 3 w1, 4 layer 1, 5 dW4, 6 dW2/db2
    uint64_t* ring_full = bars + 7;                                  // loader -> consumers, one per ring slot (32 arrivals)
    uint64_t* ring_empty = bars + 7 + RING;                          // tcgen05.commit after the last GEMM reading the slot
    uint32_t* slot = reinterpret_cast<uint32_t*>(bars + 7 + 2 * RING);
    float* xch = reinterpret_cast<float*>(sm + S::OFF_XCH);
    float* red = reinterpret_cast<float*>(sm + S::OFF_RED);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool is_mma_warp = warp == TC_COMPUTE / 32;
    const bool is_loader_warp = warp == TC_COMPUTE / 32 + 1;
    const int rw = warp & 3, half = (warp >> 2) & 1, net = (warp >> 3) & 1;
    const int r = rw * 32 + lane;
    const int u0 = half * HU;
    // One launch covers `nsteps` consecutive, equally sized minibatches (1 unless the fused tail is on): minibatch s starts at
    // mb_start + s * mb_count; every CTA has nmy >= 1 tiles in each of them (the launchers guarantee grid <= ntiles).
    const uint32_t nsteps = g.tail.enabled ? (uint32_t)g.tail.nsteps : 1u;
    const uint32_t ntiles = (g.mb_count + TC_TILE - 1) / TC_TILE;
    const uint32_t nmy = (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x;   // tiles of this CTA per minibatch (>= 1)

    // ---- prologue: barriers, TMEM, weights by TMA bulk copy ----
    TC_KSTAMP(0);
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 7; ++i) mbar_init(bars + i, 1);
#pragma unroll
        for (int i = 0; i < RING; ++i) { mbar_init(ring_full + i, 32); mbar_init(ring_empty + i, 1); }
        mbar_fence_init();
    }
    if (warp == 1) umma::tmem_alloc(slot, TC_COLS);
    if (tid == 64 && g.tail.enabled) {       // the tail's arguments -> shared memory (read after the barrier below, by everybody)
        TailCtx* c = reinterpret_cast<TailCtx*>(sm + S::OFF_CTX);
        c->tl = g.tail;
        c->grad_part = g.grad_part; c->loss_part = g.loss_part; c->packed = const_cast<float*>(g.packed); c->dbg = g.dbg;
        c->ppad = g.ppad; c->mb_count = g.mb_count; c->ent_coef = g.ent_coef; c->vf_coef = g.vf_coef;
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    if (tid == 0) {
        mbar_expect_tx(bars, (uint32_t)S::W_BYTES);
        const char* src = reinterpret_cast<const char*>(g.packed + P::TC_W2);
        for (uint32_t off = 0; off < (uint32_t)S::W_BYTES; off += 16384u) {
            const uint32_t n = (uint32_t)S::W_BYTES - off < 16384u ? (uint32_t)S::W_BYTES - off : 16384u;
            bulk_g2s(sm + S::OFF_W + off, src + off, n, bars);
        }
    }
    const uint32_t tmem = *slot;

    if (is_loader_warp) {
        // =========================== loader warp ===========================
        // lane l owns rows l, l+32, l+64, l+96 of every tile.  Indices are fetched one tile ahead of the records.
        uint32_t sidx[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) sidx[q] = tc_sample_index(g, g.mb_start, g.mb_count, blockIdx.x, ntiles, lane + 32 * q);
        uint32_t b = 0, use_par = 0;
        // the gather does not depend on the weights: the loader runs straight through all minibatches of the launch, so the
        // first tiles of minibatch s + 1 are in the ring while the fold / clip / Adam tail of minibatch s is still running
        for (uint32_t jg = 0; jg < nsteps * nmy; ++jg) {
            const uint32_t j = jg % nmy;
            float4 rv[4][OP / 4 + 1];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
#pragma unroll
                for (int c = 0; c <= OP / 4; ++c) rv[q][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                rv[q][OP / 4].w = __int_as_float(-1);                  // act < 0 marks a padding row
                if (sidx[q] != 0xFFFFFFFFu) {
                    const float4* r4 = reinterpret_cast<const float4*>(g.rec + (size_t)sidx[q] * RW);
#pragma unroll
                    for (int c = 0; c < OP / 4; ++c) rv[q][c] = __ldg(r4 + c);
                    rv[q][OP / 4] = __ldg(r4 + RW / 4 - 1);
                }
            }
            if (jg + 1 < nsteps * nmy) {
                const uint32_t jn = (jg + 1) % nmy, sn = (jg + 1) / nmy;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    sidx[q] = tc_sample_index(g, g.mb_start + sn * g.mb_count, g.mb_count, blockIdx.x + jn * gridDim.x, ntiles, lane + 32 * q);
            }
            (void)j;
            if (jg >= RING) mbar_wait(ring_empty + b, use_par ^ 1u);   // the GEMMs of tile jg - RING have released the slot
            unsigned char* obst = tOBS + b * 4096;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int row = lane + 32 * q;
                float o16[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) o16[i] = 0.0f;
#pragma unroll
                for (int i = 0; i < O; ++i) {       // obs = hi + lo to 16 mantissa bits
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
            if (++b == RING) { b = 0; use_par ^= 1u; }
        }
        __syncthreads();           // end of the kernel
        return;
    }

    if (is_mma_warp) {
        // =========================== MMA-issuer warp ===========================
        const uint32_t aW2 = smem_u32(tW2), aH1 = smem_u32(tH1), aH2 = smem_u32(tH2), aDZ = smem_u32(tDZ);
        const uint32_t aOBS = smem_u32(tOBS), aDOUT = smem_u32(tDOUT), aDZ1 = smem_u32(tDZ1);
        constexpr uint32_t ID_FWD = umma::make_idesc(128, 64, false, false);
        constexpr uint32_t ID_DH1 = umma::make_idesc(128, 64, false, true);
        constexpr uint32_t ID_W2 = umma::make_idesc(128, 128, true, true);
        constexpr uint32_t ID_N16 = umma::make_idesc(128, 16, true, true);
        const uint32_t aW1B = smem_u32(tW1B);
        constexpr uint32_t ID_L1 = umma::make_idesc(128, 64, false, false);
        // layer 1 of tile k: z1 = [obs_hi|1|obs_lo] . [W1|b1|W1]^T, K = 16, both operands K-major without swizzle
        auto issue_l1 = [&](uint32_t slot_b) {
            const uint32_t obsb = aOBS + slot_b * 4096;
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2)
                umma::mma(tmem + C_ZF + n2 * 64, umma::make_desc(obsb, 2048, 128, umma::LAYOUT_NONE),
                          umma::make_desc(aW1B + n2 * 2048, 1024, 128, umma::LAYOUT_NONE), ID_L1, 0u);
            umma::commit(bars + 4);
        };
        auto issue_fwd = [&](uint32_t k) {
            const uint32_t h1b = aH1 + (k & 1u) * 32768;      // k = running tile number of the launch
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2)
#pragma unroll
                for (int kb = 0; kb < 4; ++kb)
                    umma::mma(tmem + C_ZF + n2 * 64, umma::make_desc(h1b + n2 * 16384 + kb * 32, 16, 1024, umma::LAYOUT_SW128),
                              umma::make_desc(aW2 + n2 * 8192 + kb * 32, 16, 1024, umma::LAYOUT_SW128), ID_FWD, kb > 0);
            umma::commit(bars + 1);
        };
        uint32_t bn = 0, bn_par = 0;      // ring slot / use parity of the NEXT tile to get its layer-1 GEMM
        uint32_t bc = 0;                  // ring slot of the current tile
        for (uint32_t s = 0; s < nsteps; ++s) {
        const uint32_t kbase = s * nmy;
        mbar_wait(bars, s & 1u);   // the weight tiles of this minibatch have landed
        named_bar_sync(BAR_L1, TC_THREADS);
        mbar_wait(ring_full + bn, bn_par);
        umma::fence_after_sync();
        if (umma::elect_one()) issue_l1(bn);
        __syncwarp();
        if (++bn == RING) { bn = 0; bn_par ^= 1u; }
        named_bar_sync(BAR_FWD, TC_THREADS);
        umma::fence_after_sync();
        if (umma::elect_one()) issue_fwd(kbase);
        __syncwarp();
        for (uint32_t k = 0; k < nmy; ++k) {
            const uint32_t par = (kbase + k) & 1u, acc = k > 0 ? 1u : 0u;
            const uint32_t obsb = aOBS + bc * 4096;
            if (k + 1 < nmy) {
                named_bar_sync(BAR_L1, TC_THREADS);      // z2(k) consumed
                mbar_wait(ring_full + bn, bn_par);       // [obs|1] tile of k+1 written by the loader
                umma::fence_after_sync();
                if (umma::elect_one()) issue_l1(bn);
                __syncwarp();
                if (++bn == RING) { bn = 0; bn_par ^= 1u; }
            }
            named_bar_sync(BAR_BWD, TC_THREADS);
            umma::fence_after_sync();
            TC_STAMP(0);
            if (umma::elect_one()) {
#pragma unroll
                for (int n2 = 0; n2 < 2; ++n2)
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb)
                        umma::mma(tmem + C_DH + n2 * 64, umma::make_desc(aDZ + n2 * 16384 + kb * 32, 16, 1024, umma::LAYOUT_SW128),
                                  umma::make_desc(aW2 + n2 * 8192 + kb * 2048, 8192, 1024, umma::LAYOUT_SW128), ID_DH1, kb > 0);
                umma::commit(bars + 2);          // dh1 is all that Z(k) waits for
#ifdef DRL_TC_STAMPS
                if (g.dbg != nullptr && blockIdx.x == 0 && k < 12) g.dbg[256 + k * 16 + 6] = clock64();
#endif
            }
            __syncwarp();
            TC_STAMP(1);
            // fwd(k+1) is what X(k+1) waits for: it goes ahead of the weight-gradient GEMMs of tile k, which nobody needs
            // until late in X(k+1).  (All GEMM groups compete with the compute warps for shared-memory bandwidth -- a group
            // takes ~600 cycles alone and up to twice that with other groups queued behind it.)
            if (k + 1 < nmy) {
                named_bar_sync(BAR_FWD, TC_THREADS);
                umma::fence_after_sync();
                TC_STAMP(2);
                if (umma::elect_one()) issue_fwd(kbase + k + 1);
                __syncwarp();
                TC_STAMP(3);
            }
            if (umma::elect_one()) {
                const uint32_t h1b = aH1 + par * 32768;
#pragma unroll
                for (int kb = 0; kb < 8; ++kb)
                    umma::mma(tmem + C_W4, umma::make_desc(aH2 + kb * 2048, 16384, 1024, umma::LAYOUT_SW128),
                              umma::make_desc(aDOUT + kb * 256, 128, 2048, umma::LAYOUT_NONE), ID_N16, acc | (kb > 0));
                umma::commit(bars + 5);          // h2 and dout tiles may be overwritten (early in X(k+1))
#pragma unroll
                for (int kb = 0; kb < 8; ++kb)
                    umma::mma(tmem + C_W2, umma::make_desc(aDZ + kb * 2048, 16384, 1024, umma::LAYOUT_SW128),
                              umma::make_desc(h1b + kb * 2048, 16384, 1024, umma::LAYOUT_SW128), ID_W2, acc | (kb > 0));
#pragma unroll
                for (int kb = 0; kb < 8; ++kb)
                    umma::mma(tmem + C_B2, umma::make_desc(aDZ + kb * 2048, 16384, 1024, umma::LAYOUT_SW128),
                              umma::make_desc(obsb + kb * 256, 128, 2048, umma::LAYOUT_NONE), ID_N16, acc | (kb > 0));
                umma::commit(bars + 6);          // dz2 and h1(k) tiles may be overwritten (end of X(k+1), Y(k+1))
            }
            __syncwarp();
            named_bar_sync(BAR_W1, TC_THREADS);
            umma::fence_after_sync();
            TC_STAMP(4);
            if (umma::elect_one()) {
#pragma unroll
                for (int kb = 0; kb < 8; ++kb)
                    umma::mma(tmem + C_W1, umma::make_desc(aDZ1 + kb * 2048, 16384, 1024, umma::LAYOUT_SW128),
                              umma::make_desc(obsb + kb * 256, 128, 2048, umma::LAYOUT_NONE), ID_N16, acc | (kb > 0));
                umma::commit(bars + 3);
                umma::commit(ring_empty + bc);   // last reader of ring slot bc (tile k) is done: the loader may refill it
            }
            __syncwarp();
            TC_STAMP(5);
            if (++bc == RING) bc = 0;
        }
        }   // minibatches of the launch
        umma::fence_before_sync();
        __syncthreads();           // end of the kernel
        return;
    }

    // =========================== compute warps ===========================
    const uint32_t trow = tmem + ((uint32_t)(rw * 32) << 16);   // this thread's TMEM lane
    const float inv_m = 1.0f / (float)g.mb_count;
    const int wrow0 = net == 0 ? 0 : A;          // first head row of this net in sW4 / sB4
    const int nheads = net == 0 ? A : 1;
    uint32_t rb = 0, rb_par = 0;          // ring slot / use parity of the current tile (run on across the minibatches of the launch)

    for (uint32_t s = 0; s < nsteps; ++s) {
    const uint32_t kbase = s * nmy;              // running tile number of this minibatch's first tile: barrier phases and the h1
                                                 // double buffer continue across the minibatches of the launch
    const float adv_mean = g.adv_stats[2 * s], adv_rstd = 1.0f / (g.adv_stats[2 * s + 1] + 1e-8f);
    float lsum[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // pg, v, entropy, kl, clipfrac partial sums (half-0 threads only)
    float gb4[4] = {0.f, 0.f, 0.f, 0.f};         // head-bias gradients: actor slots 0..A-1, critic slot 3

    TC_KSTAMP(1);
    mbar_wait(bars, s & 1u);
    TC_KSTAMP(2);

    // layer-1 epilogue of tile k: z1 from TMEM -> tanh -> bf16 h1 tile (buffer k & 1), then hand fwd(k)
    auto phase0 = [&](uint32_t k) {      // k = running tile number
        mbar_wait(bars + 4, k & 1u);
        umma::fence_after_sync();
        float h[HU];
        umma::ld32(trow + C_ZF + net * 64 + u0, h);
#pragma unroll
        for (int j = 0; j < HU; ++j) h[j] = tanh_mufu(h[j]);
        store_half_row_sw128(tH1 + (k & 1u) * 32768 + net * 16384, r, half * 4, h);
        umma::fence_proxy_async();
        umma::fence_before_sync();
        named_bar_arrive(BAR_FWD, TC_THREADS);
    };

    named_bar_arrive(BAR_L1, TC_THREADS);
    phase0(kbase);
    TC_KSTAMP(3);

    for (uint32_t k = 0; k < nmy; ++k) {
        const uint32_t par = (kbase + k) & 1u;

        // ================= X(k): heads, loss, output gradients, dz2 =================
        TC_STAMP(0);
        mbar_wait(bars + 1, par);
        umma::fence_after_sync();
        TC_STAMP(1);
        {
            float h[HU];
            umma::ld32(trow + C_ZF + net * 64 + u0, h);
            if (k + 1 < nmy) {   // z2(k) is in registers: the layer-1 GEMM of tile k+1 may overwrite its TMEM columns
                umma::fence_before_sync();
                named_bar_arrive(BAR_L1, TC_THREADS);
            }
            const float* b2 = sB2 + net * H + u0;
#pragma unroll
            for (int k4 = 0; k4 < HU / 4; ++k4) {
                const float4 bb = *reinterpret_cast<const float4*>(b2 + 4 * k4);
                h[4 * k4 + 0] = tanh_mufu(h[4 * k4 + 0] + bb.x);
                h[4 * k4 + 1] = tanh_mufu(h[4 * k4 + 1] + bb.y);
                h[4 * k4 + 2] = tanh_mufu(h[4 * k4 + 2] + bb.z);
                h[4 * k4 + 3] = tanh_mufu(h[4 * k4 + 3] + bb.w);
            }
            if (k > 0) mbar_wait(bars + 5, par ^ 1u);   // dW4(k-1) has finished reading the h2 and dout tiles
            store_half_row_sw128(tH2 + net * 16384, r, half * 4, h);

            // head partial sums over this thread's 32 units, exchanged with the thread owning the other 32
            float ps[A];
#pragma unroll
            for (int a = 0; a < A; ++a) {
                ps[a] = 0.0f;
                if (a < nheads) {
                    const float* w = sW4 + (wrow0 + a) * H + u0;
                    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                    for (int k4 = 0; k4 < HU / 4; ++k4) {
                        const float4 ww = *reinterpret_cast<const float4*>(w + 4 * k4);
                        s0 = fmaf(h[4 * k4 + 0], ww.x, s0);
                        s1 = fmaf(h[4 * k4 + 1], ww.y, s1);
                        s2 = fmaf(h[4 * k4 + 2], ww.z, s2);
                        s3 = fmaf(h[4 * k4 + 3], ww.w, s3);
                    }
                    ps[a] = (s0 + s1) + (s2 + s3);
                    xch[((net * 2 + half) * 4 + a) * TC_TILE + r] = ps[a];
                }
            }
            TC_STAMP(2);
            named_bar_sync(BAR_PAIR0 + net * 4 + rw, 64);
            TC_STAMP(3);
            float out[A];
#pragma unroll
            for (int a = 0; a < A; ++a) {
                out[a] = 0.0f;
                if (a < nheads) {
                    const float po = xch[((net * 2 + (half ^ 1)) * 4 + a) * TC_TILE + r];
                    const float lo = half == 0 ? ps[a] : po, hi = half == 0 ? po : ps[a];
                    out[a] = (lo + hi) + sB4[wrow0 + a];      // identical in both threads of the pair
                }
            }
            float d[A];
#pragma unroll
            for (int a = 0; a < A; ++a) d[a] = 0.0f;
            mbar_wait(ring_full + rb, rb_par);     // long complete: the loader runs two tiles ahead
            const uint4 sc = sSCAL[rb * TC_TILE + r];
            const float rc_logp_old = __uint_as_float(sc.x), rc_adv = __uint_as_float(sc.y), rc_val_old = __uint_as_float(sc.z);
            const int rc_act = (int)sc.w;
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
                    if (half == 0) {
                        lsum[0] += fmaxf(pg1, pg2);
                        lsum[2] += ent;
                        lsum[3] += (ratio - 1.0f) - logratio;
                        lsum[4] += fabsf(ratio - 1.0f) > g.clip_coef ? 1.0f : 0.0f;
                    }
#pragma unroll
                    for (int a = 0; a < A; ++a) {
                        const float onehot = a == rc_act ? 1.0f : 0.0f;
                        d[a] = inv_m * (dpg * (onehot - p[a]) + g.ent_coef * p[a] * (lp[a] + ent));
                        if (half == 0) gb4[a] += d[a];
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
                    if (half == 0) { lsum[1] += fmaxf(vu, vcl); gb4[3] += d[0]; }
                }
            }
            if (half == 0) {   // dout row: actor -> columns 0..A-1 (chunk 0), critic -> column 8 (chunk 1)
                uint4 q = make_uint4(0u, 0u, 0u, 0u);
                if (net == 0) {
                    q.x = umma::pack_bf16(d[0], d[1]);
                    if constexpr (A > 2) q.y = umma::pack_bf16(d[2], 0.0f);
                } else {
                    q.x = umma::pack_bf16(d[0], 0.0f);
                }
                *reinterpret_cast<uint4*>(tDOUT + (size_t)net * TC_TILE * 16 + (size_t)r * 16) = q;
            }
            // dz2 = (dout . W4) * (1 - h2^2), in place
#pragma unroll
            for (int k4 = 0; k4 < HU / 4; ++k4) {
                float dh[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    if (a < nheads) {
                        const float4 ww = *reinterpret_cast<const float4*>(sW4 + (wrow0 + a) * H + u0 + 4 * k4);
                        dh[0] = fmaf(d[a], ww.x, dh[0]); dh[1] = fmaf(d[a], ww.y, dh[1]);
                        dh[2] = fmaf(d[a], ww.z, dh[2]); dh[3] = fmaf(d[a], ww.w, dh[3]);
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) h[4 * k4 + j] = dh[j] * fmaf(-h[4 * k4 + j], h[4 * k4 + j], 1.0f);
            }
            TC_STAMP(4);
            TC_STAMP(5);
            if (k > 0) mbar_wait(bars + 6, par ^ 1u);   // dW2/db2(k-1) have finished reading the dz2 and h1(k-1) tiles
            store_half_row_sw128(tDZ + net * 16384, r, half * 4, h);
        }
        umma::fence_proxy_async();
        umma::fence_before_sync();
        named_bar_arrive(BAR_BWD, TC_THREADS);
        TC_STAMP(6);

        // ================= Y(k): layer 1 of the next tile, hand fwd(k+1) (hides bwd(k)) =================
        if (k + 1 < nmy) {
            phase0(kbase + k + 1);
        }

        // ================= Z(k): dz1 = dh1 * (1 - h1^2) (hides fwd(k+1)) =================
        TC_STAMP(7);
        {
            const unsigned char* h1row = tH1 + par * 32768 + net * 16384;
            uint4 hq[4];                                   // this thread's h1 values (bf16): loaded before the wait
#pragma unroll
            for (int c = 0; c < 4; ++c) hq[c] = *reinterpret_cast<const uint4*>(h1row + umma::sw128_off(r, half * 4 + c));
            TC_STAMP(10);
            mbar_wait(bars + 2, par);
            TC_STAMP(11);
            if (k > 0) mbar_wait(bars + 3, par ^ 1u);   // w1(k-1) has finished reading tDZ1
            umma::fence_after_sync();
            TC_STAMP(8);
            float dh[HU];
            umma::ld32(trow + C_DH + net * 64 + u0, dh);
            unsigned char* dzrow = tDZ1 + net * 16384;
#pragma unroll
            for (int c = 0; c < 4; ++c) {   // 16-byte chunk at a time: h1 (bf16) in, dz1 (bf16) out
                const uint4 q = hq[c];
                const float hv[8] = {umma::bf16_lo(q.x), umma::bf16_hi(q.x), umma::bf16_lo(q.y), umma::bf16_hi(q.y),
                                     umma::bf16_lo(q.z), umma::bf16_hi(q.z), umma::bf16_lo(q.w), umma::bf16_hi(q.w)};
                float z[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) z[j] = dh[8 * c + j] * fmaf(-hv[j], hv[j], 1.0f);
                uint4 o4;
                o4.x = umma::pack_bf16(z[0], z[1]); o4.y = umma::pack_bf16(z[2], z[3]);
                o4.z = umma::pack_bf16(z[4], z[5]); o4.w = umma::pack_bf16(z[6], z[7]);
                *reinterpret_cast<uint4*>(dzrow + umma::sw128_off(r, half * 4 + c)) = o4;
            }
        }
        umma::fence_proxy_async();
        umma::fence_before_sync();
        named_bar_arrive(BAR_W1, TC_THREADS);
        TC_STAMP(9);
        if (++rb == RING) { rb = 0; rb_par ^= 1u; }
    }
    mbar_wait(bars + 3, (kbase + nmy - 1) & 1u);
    mbar_wait(bars + 5, (kbase + nmy - 1) & 1u);
    mbar_wait(bars + 6, (kbase + nmy - 1) & 1u);
    umma::fence_after_sync();
    TC_KSTAMP(4);

    // ================= epilogue: this CTA's partial gradient, canonical layout =================
    // Staged in shared memory (the tiles are dead), then copied out with coalesced stores.  A thread owns 32 consecutive
    // W2 columns of one row, so the W2 blocks are staged with the column XOR-swizzled by the row: conflict-free both ways.
    float* stage = reinterpret_cast<float*>(sm + S::OFF_H1);
    float* part = g.grad_part + (size_t)blockIdx.x * g.ppad;
    const int no = r >> 6, o = r & 63;                 // TMEM lane r = hidden unit o of net `no`
    constexpr int W2_OFF = H * O + H;                  // offset of W2 inside a net's canonical block
    if (warp < 4) {
        const int base = no * P::C_ACTOR;
        float v16[16];
        umma::ld16(trow + C_B2, v16);
        stage[base + H * O + H + H * H + o] = v16[O];   // db2
        umma::ld16(trow + C_W1, v16);
#pragma unroll
        for (int i = 0; i < O; ++i) stage[base + o * O + i] = v16[i] + v16[8 + i];   // dW1 = dz1^T . (obs_hi + obs_lo)
        stage[base + H * O + o] = v16[O];                               // db1
        umma::ld16(trow + C_W4, v16);
        if (no == 0) {
#pragma unroll
            for (int a = 0; a < A; ++a) stage[P::C_NET + a * H + o] = v16[a];   // actor head
        } else {
            stage[P::C_ACTOR + P::C_NET + o] = v16[8];                           // critic head
        }
    }
    if (no == net) {   // dW2: the diagonal 64x64 blocks of the 128x128 accumulator (warp-uniform branch)
        float v[HU];
        umma::ld32(trow + C_W2 + net * 64 + u0, v);
        float* dst = stage + net * P::C_ACTOR + W2_OFF + o * H;
#pragma unroll
        for (int i = 0; i < HU; ++i) dst[(u0 + i) ^ (o & 31)] = v[i];
    }
    // loss partial sums and head-bias gradients: fold the 512 compute threads
    {
        float vals[9] = {lsum[0], lsum[1], lsum[2], lsum[3], lsum[4], gb4[0], gb4[1], gb4[2], gb4[3]};
#pragma unroll
        for (int q = 0; q < 9; ++q) {
            const float sv = warp_sum(vals[q]);
            if (lane == 0) red[warp * 12 + q] = sv;
        }
    }
    umma::fence_before_sync();
    named_bar_sync(13, TC_COMPUTE);       // compute warps only: the issuer and the loader run on into the next minibatch
    if (tid < 9) {
        float sv = 0.0f;
#pragma unroll
        for (int w = 0; w < TC_COMPUTE / 32; ++w) sv += red[w * 12 + tid];
        if (tid < 5) g.loss_part[blockIdx.x * LOSS_TERMS + tid] = sv;
        else if (tid - 5 < A) stage[P::C_NET + A * H + (tid - 5)] = sv;              // actor head bias
        else if (tid == 8) stage[P::C_ACTOR + P::C_NET + H] = sv;                    // critic head bias
    }
    named_bar_sync(13, TC_COMPUTE);
    for (int i = tid; i < P::C_ALL; i += TC_COMPUTE) {
        const int nb = i >= P::C_ACTOR ? 1 : 0;
        const int w = i - nb * P::C_ACTOR - W2_OFF;    // index inside this net's W2 block, if 0 <= w < H*H
        int src = i;
        if (w >= 0 && w < H * H) src = i - (w & 63) + ((w & 63) ^ ((w >> 6) & 31));
        part[i] = stage[src];
    }
    TC_KSTAMP(5);
    if (g.tail.enabled) tc_tail_step<O, A>(reinterpret_cast<const TailCtx*>(sm + S::OFF_CTX), s, nsteps, sm, bars);
    }   // minibatches of the launch
    umma::fence_before_sync();
    __syncthreads();           // end of the kernel: with the issuer and the loader warp
    if (warp == 1) umma::tmem_dealloc(tmem, TC_COLS);
}

template <int O, int A, int OP, int RW>
static int launch_tc_fused(GradArgs& g, cudaStream_t st) {
    const int smem = TcSmem<O, A>::TOTAL;
    DRL_CUDA(cudaFuncSetAttribute(ppo_grad_tc_kernel<O, A, OP, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const uint32_t ntiles = (g.mb_count + TC_TILE - 1) / TC_TILE;
    int grid = sm_count();
    if (grid > MAX_GRAD_CTAS) grid = MAX_GRAD_CTAS;
    if ((uint32_t)grid > ntiles) grid = (int)ntiles;
    void* args[] = {&g};
    DRL_CUDA(cudaLaunchCooperativeKernel((const void*)ppo_grad_tc_kernel<O, A, OP, RW>, dim3(grid), dim3(GRAD_TC_BLOCK), args, (size_t)smem, st));
    return DRL_OK;
}

int launch_grad_tc_fused(const drl_net_t* net, GradArgs& g, cudaStream_t st) {
    if (net->obs_dim == 4) return launch_tc_fused<4, 2, 4, 8>(g, st);
    if (net->obs_dim == 2) return launch_tc_fused<2, 3, 4, 8>(g, st);
    return launch_tc_fused<6, 3, 8, 16>(g, st);
}

template <int O, int A, int OP, int RW>
static int launch_tc(const GradArgs& g, int P, float* grad_out, float* loss_terms_out, cudaStream_t st, int* grid_out) {
    const int smem = TcSmem<O, A>::TOTAL;
    DRL_CUDA(cudaFuncSetAttribute(ppo_grad_tc_kernel<O, A, OP, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const uint32_t ntiles = (g.mb_count + TC_TILE - 1) / TC_TILE;
    int grid = sm_count();
    if (grid > MAX_GRAD_CTAS) grid = MAX_GRAD_CTAS;
    if ((uint32_t)grid > ntiles) grid = (int)ntiles;
    ppo_grad_tc_kernel<O, A, OP, RW><<<grid, GRAD_TC_BLOCK, smem, st>>>(g);
    DRL_LAUNCH_CHECK("ppo_grad_tc_kernel");
    if (grid_out != nullptr) { *grid_out = grid; return DRL_OK; }
    return launch_grad_reduce(g, grid, P, 1, P, grad_out, loss_terms_out, st);
}

int launch_grad_tc(const drl_net_t* net, const GradArgs& g, int P, float* grad_out, float* loss_terms_out, cudaStream_t st,
                   int* grid_out) {
    if (net->obs_dim == 4) return launch_tc<4, 2, 4, 8>(g, P, grad_out, loss_terms_out, st, grid_out);
    if (net->obs_dim == 2) return launch_tc<2, 3, 4, 8>(g, P, grad_out, loss_terms_out, st, grid_out);
    return launch_tc<6, 3, 8, 16>(g, P, grad_out, loss_terms_out, st, grid_out);
}

}  // namespace drl
