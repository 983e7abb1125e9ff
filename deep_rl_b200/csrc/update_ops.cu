// update_ops.cu -- one PPO minibatch step on the GPU (deep_rl/ppo.py:159-192):
//   ppo_grad_kernel   gather records by index -> actor+critic forward -> clipped-surrogate / value /
//                     entropy loss (ppo.py:166-187) -> closed-form backward (SURVEY.md App. B.4) ->
//                     per-CTA partial gradients (FP32 CUDA-core path)
//   grad_reduce_kernel fixed-order sum of the per-CTA partials -> flat gradient + loss terms
//   clip_adam_kernel  clip_grad_norm_ + Adam (+ refresh of the packed kernel layout), ppo.py:191-192
#include "drl_h256.cuh"
#include "drl_mlp.cuh"
#include "drl_pack.cuh"
#include "drl_update.cuh"

namespace drl {

namespace h256 {
int launch_grad256(const drl_net_t* net, const GradArgs& g, int P, float* grad_out, float* loss_terms_out, void* workspace,
                   cudaStream_t st);      // update256.cu
}

constexpr int GW = 8;                 // warps per CTA
constexpr int GT = GW * 32;           // threads per CTA
constexpr int CTA_TILE = GW * TILE;   // samples per CTA tile
constexpr int DZ2_S = H1_S;           // floats: dz2 tile [net][o][e]
constexpr int DOUT_S = 64;            // floats: dout tile [net][e][4]
constexpr int WS_G = OBS_S + H1_S + DZ2_S + OUT_S + DOUT_S;

template <int O, int A>
struct GradLocal {                    // lane-local gradient accumulators (units u + 16 j of one net)
    static constexpr int N = 4 * O + 8 + 5 * A;
    float w1[UPL][O];
    float b1[UPL];
    float b2[UPL];
    float w4[A][UPL];
    float b4[A];
};

template <int O, int A, int OP, int RW>
__global__ void __launch_bounds__(GT, 1) ppo_grad_kernel(GradArgs g) {
    using P = Packed<O, A>;
    extern __shared__ __align__(128) float smem[];
    float* sw = smem;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + P::ALL);
    float* scratch = smem + P::ALL + 4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float* obs_s = scratch + warp * WS_G;
    float* h1_s = obs_s + OBS_S;
    float* dz2_s = h1_s + H1_S;
    float* out_s = dz2_s + DZ2_S;
    float* dout_s = out_s + OUT_S;
    stage_params(sw, g.packed, P::ALL, bar);

    const int net = lane >> 4, u = lane & 15;
    const float adv_mean = g.adv_stats[0], adv_std = g.adv_stats[1];
    const float inv_m = 1.0f / (float)g.mb_count;

    // phase-B ownership: dW2[net_b][o][i] patch of 4 (o) x 8 (i)
    const int net_b = warp >> 2, ob = (warp >> 1) & 1, ib = warp & 1, og = lane & 7, ig = lane >> 3;
    float acc2[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc2[a][b] = 0.0f;

    GradLocal<O, A> gl;
#pragma unroll
    for (int j = 0; j < UPL; ++j) {
#pragma unroll
        for (int i = 0; i < O; ++i) gl.w1[j][i] = 0.0f;
        gl.b1[j] = 0.0f; gl.b2[j] = 0.0f;
#pragma unroll
        for (int a = 0; a < A; ++a) gl.w4[a][j] = 0.0f;
    }
#pragma unroll
    for (int a = 0; a < A; ++a) gl.b4[a] = 0.0f;
    float s_pg = 0.f, s_v = 0.f, s_ent = 0.f, s_kl = 0.f, s_clip = 0.f;

    const uint32_t ntiles = (g.mb_count + CTA_TILE - 1) / CTA_TILE;
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // ---- A0: gather the warp's 8 sample records ----
        float logp_old = 0.f, adv = 0.f, val_old = 0.f;
        int act = 0;
        bool valid = false;
        if (lane < TILE) {
            const uint32_t pos = tile * CTA_TILE + warp * TILE + lane;
            valid = pos < g.mb_count;
            float x[OP];
#pragma unroll
            for (int i = 0; i < OP; ++i) x[i] = 0.0f;
            if (valid) {
                const uint32_t i = g.mb_start + pos;
                const size_t s = g.idx ? g.idx[i] : i;
                const float4* r4 = reinterpret_cast<const float4*>(g.rec + s * RW);
#pragma unroll
                for (int q = 0; q < OP / 4; ++q) {
                    const float4 v = __ldg(r4 + q);
                    x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
                }
                const float4 t4 = __ldg(r4 + RW / 4 - 1);
                logp_old = t4.x; adv = t4.y; val_old = t4.z; act = __float_as_int(t4.w);
            }
#pragma unroll
            for (int i = 0; i < O; ++i) obs_s[i * TILE + lane] = x[i];
        }
        __syncwarp();

        // ---- A1: forward ----
        float h2[TILE][UPL];
        mlp_forward_tile<O, A>(sw, obs_s, h1_s, out_s, lane, h2);

        // ---- A2: loss and output gradients, one sample per lane (lanes 0-7) ----
        if (lane < TILE) {
            float dl[4] = {0.f, 0.f, 0.f, 0.f};
            float dv = 0.f;
            if (valid) {
                float l[A];
#pragma unroll
                for (int a = 0; a < A; ++a) l[a] = out_s[lane * OUT_W + a];
                const float v = out_s[lane * OUT_W + 3];
                float m = l[0];
#pragma unroll
                for (int a = 1; a < A; ++a) m = fmaxf(m, l[a]);
                float se = 0.f;
#pragma unroll
                for (int a = 0; a < A; ++a) se += expf(l[a] - m);
                const float lse = m + logf(se);
                float lp[A], p[A];
                float ent = 0.f, new_logp = 0.f;
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    lp[a] = l[a] - lse;
                    p[a] = expf(lp[a]);
                    ent -= p[a] * lp[a];
                    if (a == act) new_logp = lp[a];
                }
                const float nadv = (adv - adv_mean) / (adv_std + 1e-8f);
                const float logratio = new_logp - logp_old;
                const float ratio = expf(logratio);
                const float pg1 = -nadv * ratio;
                const float pg2 = -nadv * fminf(fmaxf(ratio, 1.0f - g.clip_coef), 1.0f + g.clip_coef);
                const float dpg = pg1 >= pg2 ? pg1 : 0.0f;   // d max(pg1,pg2) / d new_logp  (= -nadv*ratio)
                const float ret = adv + val_old;             // returns = advantages + values, ppo.py:151
                const float vd = v - ret;
                const float vu = vd * vd;
                const float vc = val_old + fminf(fmaxf(v - val_old, -g.clip_coef), g.clip_coef);
                const float vcd = vc - ret;
                const float vcl = vcd * vcd;
                s_pg += fmaxf(pg1, pg2);
                s_v += fmaxf(vu, vcl);
                s_ent += ent;
                s_kl += (ratio - 1.0f) - logratio;
                s_clip += fabsf(ratio - 1.0f) > g.clip_coef ? 1.0f : 0.0f;
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    const float onehot = a == act ? 1.0f : 0.0f;
                    dl[a] = inv_m * (dpg * (onehot - p[a]) + g.ent_coef * p[a] * (lp[a] + ent));
                }
                // d max(vu, vcl)/dv, torch semantics: the clipped branch passes gradient only inside the
                // clamp range; an exact tie splits evenly between the two branches.
                const float vdiff = v - val_old;
                const float gcl = (vdiff >= -g.clip_coef && vdiff <= g.clip_coef) ? vcd : 0.0f;
                const float gv = vu > vcl ? vd : (vcl > vu ? gcl : 0.5f * (vd + gcl));
                dv = g.vf_coef * gv * inv_m;
            }
            *reinterpret_cast<float4*>(dout_s + lane * 4) = make_float4(dl[0], dl[1], dl[2], dl[3]);
            *reinterpret_cast<float4*>(dout_s + (TILE + lane) * 4) = make_float4(dv, 0.f, 0.f, 0.f);
        }
        __syncwarp();

        // ---- A3: head backward; dz2 = (dout . W4) * (1 - h2^2) ----
        {
            float d[TILE][A];
#pragma unroll
            for (int e = 0; e < TILE; ++e) {
                const float4 t4 = *reinterpret_cast<const float4*>(dout_s + (net * TILE + e) * 4);
                const float tt[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                for (int a = 0; a < A; ++a) d[e][a] = tt[a];
            }
            float dz2[TILE][UPL];
#pragma unroll
            for (int e = 0; e < TILE; ++e)
#pragma unroll
                for (int j = 0; j < UPL; ++j) dz2[e][j] = 0.0f;
#pragma unroll
            for (int a = 0; a < A; ++a) {
                const float4 w = *reinterpret_cast<const float4*>(sw + P::W4 + (net * A + a) * H + 4 * u);
                const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int e = 0; e < TILE; ++e) {
                    gl.b4[a] += d[e][a];
#pragma unroll
                    for (int j = 0; j < UPL; ++j) {
                        gl.w4[a][j] = fmaf(d[e][a], h2[e][j], gl.w4[a][j]);
                        dz2[e][j] = fmaf(d[e][a], ww[j], dz2[e][j]);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
#pragma unroll
                for (int e = 0; e < TILE; ++e) {
                    dz2[e][j] *= fmaf(-h2[e][j], h2[e][j], 1.0f);
                    gl.b2[j] += dz2[e][j];
                }
                float* row = dz2_s + (net * H + u + 16 * j) * TILE;
                *reinterpret_cast<float4*>(row) = make_float4(dz2[0][j], dz2[1][j], dz2[2][j], dz2[3][j]);
                *reinterpret_cast<float4*>(row + 4) = make_float4(dz2[4][j], dz2[5][j], dz2[6][j], dz2[7][j]);
            }
        }
        __syncwarp();

        // ---- A4: dh1 = dz2 . W2 ; dz1 = dh1 * (1 - h1^2) ; layer-1 weight gradients ----
        {
            float acc[TILE][UPL];
#pragma unroll
            for (int e = 0; e < TILE; ++e)
#pragma unroll
                for (int j = 0; j < UPL; ++j) acc[e][j] = 0.0f;
            const float* wp = sw + P::W2P + net * H * H + 4 * u;
            const float* ap = dz2_s + net * H * TILE;
#pragma unroll 8
            for (int o = 0; o < H; ++o) {
                const float4 w = *reinterpret_cast<const float4*>(wp + o * H);
                const float4 x0 = *reinterpret_cast<const float4*>(ap + o * TILE);
                const float4 x1 = *reinterpret_cast<const float4*>(ap + o * TILE + 4);
                const float xs[TILE] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
                for (int e = 0; e < TILE; ++e) {
                    acc[e][0] = fmaf(xs[e], w.x, acc[e][0]);
                    acc[e][1] = fmaf(xs[e], w.y, acc[e][1]);
                    acc[e][2] = fmaf(xs[e], w.z, acc[e][2]);
                    acc[e][3] = fmaf(xs[e], w.w, acc[e][3]);
                }
            }
            float xo[O][TILE];
#pragma unroll
            for (int i = 0; i < O; ++i) {
                const float4 x0 = *reinterpret_cast<const float4*>(obs_s + i * TILE);
                const float4 x1 = *reinterpret_cast<const float4*>(obs_s + i * TILE + 4);
                xo[i][0] = x0.x; xo[i][1] = x0.y; xo[i][2] = x0.z; xo[i][3] = x0.w;
                xo[i][4] = x1.x; xo[i][5] = x1.y; xo[i][6] = x1.z; xo[i][7] = x1.w;
            }
#pragma unroll
            for (int j = 0; j < UPL; ++j) {
                const float* row = h1_s + (net * H + u + 16 * j) * TILE;
                const float4 a0 = *reinterpret_cast<const float4*>(row);
                const float4 a1 = *reinterpret_cast<const float4*>(row + 4);
                const float hv[TILE] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                for (int e = 0; e < TILE; ++e) {
                    const float dz1 = acc[e][j] * fmaf(-hv[e], hv[e], 1.0f);
                    gl.b1[j] += dz1;
#pragma unroll
                    for (int i = 0; i < O; ++i) gl.w1[j][i] = fmaf(dz1, xo[i][e], gl.w1[j][i]);
                }
            }
        }
        __syncthreads();

        // ---- B: dW2[o][i] += sum over the CTA's 64 samples of dz2[s][o] * h1[s][i] ----
#pragma unroll 1
        for (int w = 0; w < GW; ++w) {
            const float* hs = scratch + w * WS_G + OBS_S + net_b * H * TILE;
            const float* ds = hs + H1_S;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                float4 dz[4], hh[8];
#pragma unroll
                for (int jo = 0; jo < 4; ++jo)
                    dz[jo] = *reinterpret_cast<const float4*>(ds + (ob * 32 + og + 8 * jo) * TILE + 4 * q);
#pragma unroll
                for (int ii = 0; ii < 8; ++ii)
                    hh[ii] = *reinterpret_cast<const float4*>(hs + (ib * 32 + ig + 4 * ii) * TILE + 4 * q);
#pragma unroll
                for (int jo = 0; jo < 4; ++jo)
#pragma unroll
                    for (int ii = 0; ii < 8; ++ii)
                        acc2[jo][ii] = fmaf(dz[jo].w, hh[ii].w, fmaf(dz[jo].z, hh[ii].z,
                                       fmaf(dz[jo].y, hh[ii].y, fmaf(dz[jo].x, hh[ii].x, acc2[jo][ii]))));
            }
        }
        __syncthreads();
    }

    // ---- epilogue: per-CTA partial gradient in canonical layout ----
    float* part = g.grad_part + (size_t)blockIdx.x * g.ppad;
    {
        const int nb = net_b * P::C_ACTOR + H * O + H;   // canonical offset of W2 of net_b
#pragma unroll
        for (int jo = 0; jo < 4; ++jo)
#pragma unroll
            for (int ii = 0; ii < 8; ++ii)
                part[nb + (ob * 32 + og + 8 * jo) * H + (ib * 32 + ig + 4 * ii)] = acc2[jo][ii];
    }
    // lane-local accumulators: fold the 8 warps through shared memory (scratch is free now)
    constexpr int NL = GradLocal<O, A>::N;
    float* red = scratch;   // [GW][32][NL]
    {
        float* mine = red + (warp * 32 + lane) * NL;
        int k = 0;
#pragma unroll
        for (int j = 0; j < UPL; ++j)
#pragma unroll
            for (int i = 0; i < O; ++i) mine[k++] = gl.w1[j][i];
#pragma unroll
        for (int j = 0; j < UPL; ++j) mine[k++] = gl.b1[j];
#pragma unroll
        for (int j = 0; j < UPL; ++j) mine[k++] = gl.b2[j];
#pragma unroll
        for (int a = 0; a < A; ++a)
#pragma unroll
            for (int j = 0; j < UPL; ++j) mine[k++] = gl.w4[a][j];
#pragma unroll
        for (int a = 0; a < A; ++a) mine[k++] = gl.b4[a];
    }
    __syncthreads();
    for (int item = tid; item < 32 * NL; item += GT) {
        const int ln = item / NL, k = item % NL;
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < GW; ++w) s += red[(w * 32 + ln) * NL + k];
        const int nt = ln >> 4, uu = ln & 15;
        const int base = nt * P::C_ACTOR;
        const int nout = nt == 0 ? A : 1;
        int canon = -1;
        if (k < UPL * O) {
            const int j = k / O, i = k % O;
            canon = base + (uu + 16 * j) * O + i;
        } else if (k < UPL * O + UPL) {
            canon = base + H * O + (uu + 16 * (k - UPL * O));
        } else if (k < UPL * O + 2 * UPL) {
            canon = base + H * O + H + H * H + (uu + 16 * (k - UPL * O - UPL));
        } else if (k < UPL * O + 2 * UPL + A * UPL) {
            const int kk = k - (UPL * O + 2 * UPL);
            const int a = kk / UPL, j = kk % UPL;
            if (a < nout) canon = base + P::C_NET + a * H + (uu + 16 * j);
        } else {
            const int a = k - (UPL * O + 2 * UPL + A * UPL);
            if (uu == 0 && a < nout) canon = base + P::C_NET + nout * H + a;
        }
        if (canon >= 0) part[canon] = s;
    }
    // loss-term partial sums
    __shared__ float lsum[GW][5];
    {
        const float t0 = warp_sum(s_pg), t1 = warp_sum(s_v), t2 = warp_sum(s_ent), t3 = warp_sum(s_kl), t4 = warp_sum(s_clip);
        if (lane == 0) { lsum[warp][0] = t0; lsum[warp][1] = t1; lsum[warp][2] = t2; lsum[warp][3] = t3; lsum[warp][4] = t4; }
    }
    __syncthreads();
    if (tid < 5) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < GW; ++w) s += lsum[w][tid];
        g.loss_part[blockIdx.x * LOSS_TERMS + tid] = s;
    }
}

// Lanes 0-4 of one warp each fold one loss term over the `nrows` per-CTA partials in row order, lane 0 then stores the
// LOSS_TERMS row.  The five shuffles are written out: as an unrolled loop they lead nvcc to unroll the fold loop 4x, not 16x.
__device__ __forceinline__ void fold_loss_terms(const float* __restrict__ loss_part, int nrows, uint32_t mb_count, float ent_coef,
                                                float vf_coef, float* __restrict__ loss_terms_out) {
    float t = 0.f;
    for (int c = 0; c < nrows; ++c) t += __ldcg(loss_part + c * LOSS_TERMS + threadIdx.x);
    const float sums[5] = {__shfl_sync(0x1fu, t, 0), __shfl_sync(0x1fu, t, 1), __shfl_sync(0x1fu, t, 2), __shfl_sync(0x1fu, t, 3),
                           __shfl_sync(0x1fu, t, 4)};
    if (threadIdx.x == 0) store_loss_terms(loss_terms_out, sums, mb_count, ent_coef, vf_coef);
}

// Sum the per-CTA partials in a fixed order (deterministic) and finish the loss terms.  blockDim = (32, 8): thread (x, y)
// folds slice y of parameter p's rows (fold_partials) with independent loads in flight, then the 8 slices are added through
// shared memory in slice order.  Row selection (STRIDE, critic0): launch_grad_reduce.  The stride is a template parameter:
// with a constant trip-count divisor the compiler unrolls the fold and keeps more loads in flight.
template <int STRIDE>
__global__ void __launch_bounds__(256) grad_reduce_kernel(const float* __restrict__ grad_part, const float* __restrict__ loss_part,
                                                           int nrows, int ppad, int P, int critic0, uint32_t mb_count, float ent_coef,
                                                           float vf_coef, float* __restrict__ grad_out, float* __restrict__ loss_terms_out) {
    __shared__ float sh[8][33];
    const int p = blockIdx.x * 32 + threadIdx.x;
    float s = 0.0f;
    if (p < P) s = fold_partials(grad_part, ppad, p, (p >= critic0 ? 1 : 0) + STRIDE * threadIdx.y, STRIDE, nrows);
    sh[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && p < P) {
        float t = sh[0][threadIdx.x];
#pragma unroll
        for (int y = 1; y < 8; ++y) t += sh[y][threadIdx.x];
        grad_out[p] = t;
    }
    if (blockIdx.x == 0 && threadIdx.y == 1 && threadIdx.x < 5 && loss_terms_out != nullptr)
        fold_loss_terms(loss_part, nrows, mb_count, ent_coef, vf_coef, loss_terms_out);
}

// clip_grad_norm_ + Adam.  Every CTA recomputes the global norm from the (L2-resident) gradient in
// the same order, so no grid-wide synchronisation is needed and all CTAs agree bit-for-bit.
template <int O, int A, int HID>
__device__ __forceinline__ void packed_store_any(float* __restrict__ packed, int i, float v) {
    if constexpr (HID == 256) h256::packed_store256<O, A>(packed, i, v);
    else packed_store<O, A>(packed, i, v);
}

template <int O, int A, int HID = 64>
__global__ void __launch_bounds__(256) clip_adam_kernel(AdamArgs a) {
    __shared__ double sh[8];
    __shared__ float s_coef;
    double ss = 0.0;
    {   // 16-byte loads, four independent partial sums per thread: the whole gradient is read in ~9 round trips
        const float4* g4 = reinterpret_cast<const float4*>(a.grad);
        const int n4 = a.P / 4;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll 4
        for (int i = threadIdx.x; i < n4; i += 256) {
            const float4 q = __ldcg(g4 + i);
            const double x = (double)(q.x * a.grad_scale), y = (double)(q.y * a.grad_scale);
            const double z = (double)(q.z * a.grad_scale), w = (double)(q.w * a.grad_scale);
            s0 = fma(x, x, s0); s1 = fma(y, y, s1); s2 = fma(z, z, s2); s3 = fma(w, w, s3);
        }
        ss = (s0 + s1) + (s2 + s3);
        for (int i = n4 * 4 + threadIdx.x; i < a.P; i += 256) {
            const double gv = (double)(a.grad[i] * a.grad_scale);
            ss = fma(gv, gv, ss);
        }
    }
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sh[w];
        s_coef = clip_coef(t, a);
    }
    __syncthreads();
    const float coef = s_coef;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.P) return;
    const float gsc = (a.grad[i] * a.grad_scale) * coef;
    float m = a.m[i], v = a.v[i], p = a.params[i];
    adam_apply(gsc, m, v, p, a.om_beta1, a.beta2, a.om_beta2, a.eps, a.neg_step_size, a.bc2_sqrt);
    a.m[i] = m; a.v[i] = v; a.params[i] = p;
    if (a.packed != nullptr) packed_store_any<O, A, HID>(a.packed, i, p);
}

// Single-GPU tail of a minibatch step in ONE cooperative launch: fixed-order fold of the `nparts` per-CTA partial
// gradients, global-norm clip and Adam (+ packed-layout refresh), with the arguments of the tensor-core fused step (g.tail).
// blockDim = (32, 8): a CTA owns 32 parameters, thread (x, y) folds slice y of the partials; after a grid-wide barrier on
// tail.ctr[0] (all CTAs are co-resident: cooperative launch) every CTA sums the per-CTA squared norms in the same order and
// applies Adam to its 32 parameters.
template <int O, int A>
__global__ void __launch_bounds__(256) reduce_clip_adam_kernel(const __grid_constant__ GradArgs g, int nparts) {
    __shared__ float sh[8][33];
    __shared__ double shd[32];
    __shared__ float s_coef;
    const TailArgs& tl = g.tail;
    const AdamArgs& a = tl.a;
    uint32_t* const arrive = tl.ctr;
    uint32_t* const depart = tl.ctr + 3;
    const int P = a.P;
    const int p = blockIdx.x * 32 + threadIdx.x;
    float sacc = 0.0f;
    if (p < P) sacc = fold_partials(g.grad_part, g.ppad, p, threadIdx.y, 1, nparts);
    sh[threadIdx.y][threadIdx.x] = sacc;
    __syncthreads();
    float gval = 0.0f;
    if (threadIdx.y == 0) {
        float t = sh[0][threadIdx.x];
#pragma unroll
        for (int y = 1; y < 8; ++y) t += sh[y][threadIdx.x];
        gval = p < P ? t : 0.0f;
        if (p < P) tl.grad_out[p] = gval;
        const double gs = (double)(gval * a.grad_scale);
        shd[threadIdx.x] = gs * gs;
    }
    if (blockIdx.x == 0 && threadIdx.y == 1 && threadIdx.x < 5 && tl.loss_terms_out != nullptr)
        fold_loss_terms(g.loss_part, nparts, g.mb_count, g.ent_coef, g.vf_coef, tl.loss_terms_out);
    __syncthreads();
    // ---- grid-wide barrier, then every CTA folds the per-CTA squared norms in the same (lane-strided) order ----
    if (threadIdx.y == 0) {
        double t = shd[threadIdx.x];
        t = warp_sum(t);
        if (threadIdx.x == 0) {
            tl.cta_sumsq[blockIdx.x] = t;
            __threadfence();
            atomicAdd(arrive, 1u);
            while (*reinterpret_cast<volatile uint32_t*>(arrive) < gridDim.x) { }
            __threadfence();
        }
        __syncwarp();
        double tot = 0.0;
        for (unsigned i = threadIdx.x; i < gridDim.x; i += 32) tot += __ldcg(tl.cta_sumsq + i);
        tot = warp_sum(tot);
        if (threadIdx.x == 0) s_coef = clip_coef(tot, a);
    }
    __syncthreads();
    if (threadIdx.y == 0 && p < P) {
        const float gsc = (gval * a.grad_scale) * s_coef;
        float m = a.m[p], v = a.v[p], w = a.params[p];
        adam_apply(gsc, m, v, w, a.om_beta1, a.beta2, a.om_beta2, a.eps, a.neg_step_size, a.bc2_sqrt);
        a.m[p] = m; a.v[p] = v; a.params[p] = w;
        if (a.packed != nullptr) packed_store<O, A>(a.packed, p, w);
    }
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        __threadfence();
        if (atomicAdd(depart, 1u) == gridDim.x - 1) { *arrive = 0u; *depart = 0u; }   // re-arm (stream-ordered)
    }
}

template <int O, int A, int OP, int RW>
int launch_grad(const GradArgs& g, int P, float* grad_out, float* loss_terms_out, cudaStream_t st, int* grid_out) {
    const size_t smem = sizeof(float) * (Packed<O, A>::ALL + 4 + GW * WS_G);
    DRL_CUDA(cudaFuncSetAttribute(ppo_grad_kernel<O, A, OP, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t ntiles = (g.mb_count + CTA_TILE - 1) / CTA_TILE;
    int grid = sm_count();
    if (grid > MAX_GRAD_CTAS) grid = MAX_GRAD_CTAS;
    if ((uint32_t)grid > ntiles) grid = (int)ntiles;
    ppo_grad_kernel<O, A, OP, RW><<<grid, GT, smem, st>>>(g);
    DRL_LAUNCH_CHECK("ppo_grad_kernel");
    if (grid_out != nullptr) { *grid_out = grid; return DRL_OK; }   // caller folds the partials itself
    return launch_grad_reduce(g, grid, P, 1, P, grad_out, loss_terms_out, st);
}

template <int HID>
static void launch_clip_adam(const drl_net_t* net, const AdamArgs& a, cudaStream_t st) {
    const int blocks = (a.P + 255) / 256;
    if (net->obs_dim == 4) clip_adam_kernel<4, 2, HID><<<blocks, 256, 0, st>>>(a);
    else if (net->obs_dim == 2) clip_adam_kernel<2, 3, HID><<<blocks, 256, 0, st>>>(a);
    else clip_adam_kernel<6, 3, HID><<<blocks, 256, 0, st>>>(a);
}

int launch_grad_reduce(const GradArgs& g, int nrows, int P, int stride, int critic0, float* grad_out, float* loss_terms_out,
                       cudaStream_t st) {
    const auto kernel = stride == 2 ? grad_reduce_kernel<2> : grad_reduce_kernel<1>;
    kernel<<<(P + 31) / 32, dim3(32, 8), 0, st>>>(g.grad_part, g.loss_part, nrows, g.ppad, P, critic0, g.mb_count, g.ent_coef,
                                                  g.vf_coef, grad_out, loss_terms_out);
    DRL_LAUNCH_CHECK("grad_reduce_kernel");
    return DRL_OK;
}

}  // namespace drl

using namespace drl;

extern "C" {

static int run_grad(const drl_net_t* net, const float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                    uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* grad_out, float* loss_terms_out,
                    void* workspace, size_t workspace_bytes, uint32_t flags, cudaStream_t st, GradArgs* g_out, int* grid_out) {
    DRL_REQUIRE(packed && rec && adv_stats && coef && grad_out && workspace, "minibatch gradient: NULL pointer");
    DRL_REQUIRE(mb_count > 0, "minibatch gradient: empty minibatch");
    const int P = (int)drl_param_count(net);
    const WorkspaceLayout w = workspace_layout(P, net->hidden);
    DRL_REQUIRE(workspace_bytes >= w.total, "minibatch gradient: workspace %zu < %zu bytes", workspace_bytes, w.total);
    GradArgs g;
    g.packed = packed; g.rec = rec; g.idx = idx; g.mb_start = mb_start; g.mb_count = mb_count; g.adv_stats = adv_stats;
    g.clip_coef = coef->clip_coef; g.ent_coef = coef->ent_coef; g.vf_coef = coef->vf_coef;
    g.grad_part = reinterpret_cast<float*>((char*)workspace + w.grad_partials);
    g.loss_part = reinterpret_cast<float*>((char*)workspace + w.loss_partials);
    g.ppad = w.ppad;
    g.dbg = getenv("DRL_TC_DEBUG") ? reinterpret_cast<long long*>((char*)workspace + w.debug) : nullptr;
    g.tail.enabled = 0;
    g.tail.ctrl = nullptr; g.tail.ordinal = 0; g.tail.nsteps = 1;
    if (g_out) { *g_out = g; if (grid_out == nullptr) return DRL_OK; }   // arguments only
    if (net->hidden == 256) {
        DRL_REQUIRE(flags & DRL_GRAD_TENSOR_CORES, "minibatch gradient: hidden=256 exists on the tensor-core path only");
        DRL_REQUIRE(grid_out == nullptr, "minibatch gradient: hidden=256 has no fused fold");
        return h256::launch_grad256(net, g, P, grad_out, loss_terms_out, workspace, st);
    }
    if (flags & DRL_GRAD_TENSOR_CORES) return launch_grad_tc(net, g, P, grad_out, loss_terms_out, st, grid_out);
    if (net->obs_dim == 4) return launch_grad<4, 2, 4, 8>(g, P, grad_out, loss_terms_out, st, grid_out);
    if (net->obs_dim == 2) return launch_grad<2, 3, 4, 8>(g, P, grad_out, loss_terms_out, st, grid_out);
    return launch_grad<6, 3, 8, 16>(g, P, grad_out, loss_terms_out, st, grid_out);
}

static void fill_adam(AdamArgs& a, const drl_net_t* net, float* params, const float* grad, float* exp_avg, float* exp_avg_sq,
                      int64_t step, double lr, double beta1, double beta2, double eps, double max_grad_norm, double grad_scale,
                      float* packed_out, float* norm_out) {
    a.params = params; a.grad = grad; a.m = exp_avg; a.v = exp_avg_sq; a.packed = packed_out; a.norm_out = norm_out;
    a.P = (int)drl_param_count(net);
    a.grad_scale = (float)grad_scale; a.max_norm = (float)max_grad_norm;
    a.beta2 = (float)beta2; a.om_beta1 = (float)(1.0 - beta1); a.om_beta2 = (float)(1.0 - beta2); a.eps = (float)eps;
    const AdamScalars s = adam_scalars(step, lr, beta1, beta2);
    a.neg_step_size = s.neg_step_size;
    a.bc2_sqrt = s.bc2_sqrt;
}

int drl_ppo_minibatch_grad(const drl_net_t* net, const float* packed, const float* rec, const uint32_t* idx,
                           uint32_t mb_start, uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef,
                           float* grad_out, float* loss_terms_out, void* workspace, size_t workspace_bytes, uint32_t flags, void* stream) {
    int rc = check_net(net);
    if (rc != DRL_OK) return rc;
    return run_grad(net, packed, rec, idx, mb_start, mb_count, adv_stats, coef, grad_out, loss_terms_out, workspace, workspace_bytes,
                    flags, as_stream(stream), nullptr, nullptr);
}

static int minibatch_update_impl(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                                 uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params, float* grad_out,
                                 float* exp_avg, float* exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                                 double max_grad_norm, float* loss_terms_out, float* norm_out, void* workspace, size_t workspace_bytes,
                                 uint32_t flags, const drl_comm_t* comm, void* stream, const drl_ctrl_t* ctrl = nullptr, int ordinal = 0,
                                 int num_steps = 1) {
    int rc = check_net(net);
    if (rc != DRL_OK) return rc;
    if (net->hidden != H) { set_error("drl_ppo_minibatch_update: hidden=%d has no fused step (use drl_ppo_minibatch_grad + drl_clip_adam)", net->hidden); return DRL_ERR_UNSUPPORTED; }
    DRL_REQUIRE(params && exp_avg && exp_avg_sq, "drl_ppo_minibatch_update: NULL pointer");
    DRL_REQUIRE(step >= 1, "drl_ppo_minibatch_update: step=%lld must be >= 1", (long long)step);
    DRL_REQUIRE(num_steps >= 1 && num_steps <= DRL_MAX_STEPS_PER_LAUNCH, "drl_ppo_minibatch_update: num_steps=%d (1..%d)", num_steps,
                DRL_MAX_STEPS_PER_LAUNCH);
    DRL_REQUIRE(num_steps == 1 || (flags & DRL_GRAD_TENSOR_CORES), "drl_ppo_minibatch_update: num_steps > 1 needs the tensor-core path");
    DRL_REQUIRE(ctrl == nullptr || ordinal + num_steps <= DRL_CTRL_MAX_STEPS, "drl_ppo_minibatch_update: ordinal %d + %d steps > %d", ordinal,
                num_steps, DRL_CTRL_MAX_STEPS);
    const bool tc = flags & DRL_GRAD_TENSOR_CORES;
    DRL_REQUIRE(tc || comm == nullptr, "drl_ppo_minibatch_update: the fp32 path has no fused multi-GPU form");
    cudaStream_t st = as_stream(stream);
    GradArgs g;
    int grid = 0;
    // tcgen05: arguments only, the gradient and its tail are one cooperative launch (gradient + fold + [peer all-reduce] + clip
    // + Adam).  fp32: launches the gradient kernel; reduce_clip_adam_kernel (fold + clip + Adam) then reads the same g.tail.
    rc = run_grad(net, packed, rec, idx, mb_start, mb_count, adv_stats, coef, grad_out, loss_terms_out, workspace, workspace_bytes,
                  flags, st, &g, tc ? nullptr : &grid);
    if (rc != DRL_OK) return rc;
    const WorkspaceLayout w = workspace_layout(drl_param_count(net));
    const int world = comm ? comm->world : 1;
    g.tail.enabled = 1;
    fill_adam(g.tail.a, net, params, grad_out, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, max_grad_norm, 1.0 / world, packed,
              norm_out);
    g.tail.grad_out = grad_out; g.tail.loss_terms_out = loss_terms_out;
    g.tail.cta_sumsq = reinterpret_cast<double*>((char*)workspace + w.cta_sumsq);
    g.tail.ctr = reinterpret_cast<uint32_t*>((char*)workspace + w.counters) + 8;
    g.tail.world = world; g.tail.rank = comm ? comm->rank : 0; g.tail.seq = comm ? comm->seq : 0;
    g.tail.error_flag = comm ? comm->error_flag : nullptr;
    g.tail.ctrl = ctrl; g.tail.ordinal = ordinal;
    g.tail.nsteps = num_steps;
    for (int sidx = 0; sidx < num_steps; ++sidx) {      // by-value Adam scalars of optimizer steps step .. step + num_steps - 1
        const AdamScalars s = adam_scalars(step + sidx, lr, beta1, beta2);
        g.tail.neg_step_size_s[sidx] = s.neg_step_size;
        g.tail.bc2_sqrt_s[sidx] = s.bc2_sqrt;
    }
    for (int r = 0; r < DRL_MAX_RANKS; ++r)
        g.tail.peer[r] = (comm && r < world) ? reinterpret_cast<unsigned char*>(comm->peer[r]) : nullptr;
    if (tc) return launch_grad_tc_fused(net, g, st);
    const int blocks = (g.tail.a.P + 31) / 32;
    DRL_REQUIRE(blocks <= 1024, "drl_ppo_minibatch_update: %d parameters exceed the squared-norm scratch", g.tail.a.P);
    void* args[] = {&g, &grid};
    const void* fn = net->obs_dim == 4 ? (const void*)reduce_clip_adam_kernel<4, 2>
                     : net->obs_dim == 2 ? (const void*)reduce_clip_adam_kernel<2, 3> : (const void*)reduce_clip_adam_kernel<6, 3>;
    DRL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(blocks), dim3(32, 8), args, 0, st));
    return DRL_OK;
}

int drl_ppo_minibatch_update(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                             uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params, float* grad_out,
                             float* exp_avg, float* exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                             double max_grad_norm, float* loss_terms_out, float* norm_out, void* workspace, size_t workspace_bytes,
                             uint32_t flags, int32_t num_steps, void* stream) {
    return minibatch_update_impl(net, packed, rec, idx, mb_start, mb_count, adv_stats, coef, params, grad_out, exp_avg, exp_avg_sq, step,
                                 lr, beta1, beta2, eps, max_grad_norm, loss_terms_out, norm_out, workspace, workspace_bytes, flags,
                                 nullptr, stream, nullptr, 0, num_steps);
}

int drl_ppo_minibatch_update_dist(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                                  uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params,
                                  float* grad_out, float* exp_avg, float* exp_avg_sq, int64_t step, double lr, double beta1,
                                  double beta2, double eps, double max_grad_norm, float* loss_terms_out, float* norm_out,
                                  void* workspace, size_t workspace_bytes, uint32_t flags, const drl_comm_t* comm, int32_t num_steps,
                                  void* stream) {
    DRL_REQUIRE(comm != nullptr, "drl_ppo_minibatch_update_dist: comm is NULL");
    DRL_REQUIRE(comm->world >= 1 && comm->world <= DRL_MAX_RANKS && comm->rank >= 0 && comm->rank < comm->world,
                "drl_ppo_minibatch_update_dist: world=%d rank=%d", comm->world, comm->rank);
    DRL_REQUIRE(flags & DRL_GRAD_TENSOR_CORES, "drl_ppo_minibatch_update_dist: tensor-core path only");
    for (int r = 0; r < comm->world; ++r) DRL_REQUIRE(comm->peer[r] != nullptr, "drl_ppo_minibatch_update_dist: peer[%d] is NULL", r);
    return minibatch_update_impl(net, packed, rec, idx, mb_start, mb_count, adv_stats, coef, params, grad_out, exp_avg, exp_avg_sq, step,
                                 lr, beta1, beta2, eps, max_grad_norm, loss_terms_out, norm_out, workspace, workspace_bytes, flags,
                                 comm, stream, nullptr, 0, num_steps);
}

int drl_ppo_minibatch_update_ctl(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                                 uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params,
                                 float* grad_out, float* exp_avg, float* exp_avg_sq, const drl_ctrl_t* ctrl, int32_t ordinal,
                                 double beta1, double beta2, double eps, double max_grad_norm, float* loss_terms_out,
                                 float* norm_out, void* workspace, size_t workspace_bytes, uint32_t flags, const drl_comm_t* comm,
                                 int32_t num_steps, void* stream) {
    DRL_REQUIRE(ctrl != nullptr, "drl_ppo_minibatch_update_ctl: ctrl is NULL");
    DRL_REQUIRE(ordinal >= 0 && ordinal < DRL_CTRL_MAX_STEPS, "drl_ppo_minibatch_update_ctl: ordinal=%d", ordinal);
    DRL_REQUIRE(flags & DRL_GRAD_TENSOR_CORES, "drl_ppo_minibatch_update_ctl: tensor-core path only");
    if (comm != nullptr) {
        DRL_REQUIRE(comm->world >= 1 && comm->world <= DRL_MAX_RANKS && comm->rank >= 0 && comm->rank < comm->world,
                    "drl_ppo_minibatch_update_ctl: world=%d rank=%d", comm->world, comm->rank);
        for (int r = 0; r < comm->world; ++r) DRL_REQUIRE(comm->peer[r] != nullptr, "drl_ppo_minibatch_update_ctl: peer[%d] is NULL", r);
    }
    // step = 1 / lr = 0 only feed the by-value Adam scalars, which the kernel replaces with ctrl's
    return minibatch_update_impl(net, packed, rec, idx, mb_start, mb_count, adv_stats, coef, params, grad_out, exp_avg, exp_avg_sq, 1,
                                 0.0, beta1, beta2, eps, max_grad_norm, loss_terms_out, norm_out, workspace, workspace_bytes, flags,
                                 comm, stream, ctrl, ordinal, num_steps);
}

__global__ void ctrl_set_kernel(drl_ctrl_t* dst, drl_ctrl_t v) {
    if (threadIdx.x == 0) { dst->env_step = v.env_step; dst->epoch_ctr = v.epoch_ctr; dst->comm_seq = v.comm_seq; dst->adam_step = v.adam_step; }
    if (threadIdx.x < DRL_CTRL_MAX_STEPS) { dst->neg_step_size[threadIdx.x] = v.neg_step_size[threadIdx.x]; dst->bc2_sqrt[threadIdx.x] = v.bc2_sqrt[threadIdx.x]; }
}

int drl_ctrl_set(drl_ctrl_t* ctrl, uint64_t env_step, uint32_t epoch_ctr, uint32_t comm_seq, int64_t adam_step, int32_t n_steps,
                 double lr, double beta1, double beta2, void* stream) {
    DRL_REQUIRE(ctrl != nullptr, "drl_ctrl_set: ctrl is NULL");
    DRL_REQUIRE(n_steps >= 0 && n_steps <= DRL_CTRL_MAX_STEPS, "drl_ctrl_set: n_steps=%d (max %d)", n_steps, DRL_CTRL_MAX_STEPS);
    DRL_REQUIRE(adam_step >= 0, "drl_ctrl_set: adam_step=%lld", (long long)adam_step);
    drl_ctrl_t v;
    memset(&v, 0, sizeof(v));
    v.env_step = env_step; v.epoch_ctr = epoch_ctr; v.comm_seq = comm_seq; v.adam_step = adam_step;
    for (int k = 0; k < n_steps; ++k) {      // optimizer steps adam_step + 1 ... adam_step + n_steps
        const AdamScalars s = adam_scalars(adam_step + k + 1, lr, beta1, beta2);
        v.neg_step_size[k] = s.neg_step_size;
        v.bc2_sqrt[k] = s.bc2_sqrt;
    }
    ctrl_set_kernel<<<1, DRL_CTRL_MAX_STEPS, 0, as_stream(stream)>>>(ctrl, v);
    DRL_LAUNCH_CHECK("ctrl_set_kernel");
    return DRL_OK;
}

size_t drl_comm_bytes(const drl_net_t* net) {
    if (check_net(net) != DRL_OK) return 0;
    return comm_layout(drl_param_count(net)).total;
}
int drl_comm_alloc(size_t bytes, void** dev_ptr_out, void* ipc_handle_out) {
    DRL_REQUIRE(dev_ptr_out && ipc_handle_out && bytes > 0, "drl_comm_alloc: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    void* p = nullptr;
    DRL_CUDA(cudaMalloc(&p, bytes));
    DRL_CUDA(cudaMemset(p, 0, bytes));
    DRL_CUDA(cudaDeviceSynchronize());
    DRL_CUDA(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(ipc_handle_out), p));
    *dev_ptr_out = p;
    return DRL_OK;
}
int drl_comm_open(const void* ipc_handle, void** peer_ptr_out) {
    DRL_REQUIRE(ipc_handle && peer_ptr_out, "drl_comm_open: NULL pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, sizeof(h));
    DRL_CUDA(cudaIpcOpenMemHandle(peer_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return DRL_OK;
}
int drl_comm_close(void* peer_ptr) {
    DRL_REQUIRE(peer_ptr, "drl_comm_close: NULL pointer");
    DRL_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return DRL_OK;
}
int drl_comm_free(void* dev_ptr) {
    DRL_REQUIRE(dev_ptr, "drl_comm_free: NULL pointer");
    DRL_CUDA(cudaFree(dev_ptr));
    return DRL_OK;
}

int drl_clip_adam(const drl_net_t* net, float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t step,
                  double lr, double beta1, double beta2, double eps, double max_grad_norm, double grad_scale,
                  float* packed_out, float* norm_out, void* stream) {
    int rc = check_net(net);
    if (rc != DRL_OK) return rc;
    DRL_REQUIRE(params && grad && exp_avg && exp_avg_sq, "drl_clip_adam: NULL pointer");
    DRL_REQUIRE(step >= 1, "drl_clip_adam: step=%lld must be >= 1", (long long)step);
    AdamArgs a;
    fill_adam(a, net, params, grad, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, max_grad_norm, grad_scale, packed_out, norm_out);
    if (net->hidden == 256) launch_clip_adam<256>(net, a, as_stream(stream));
    else launch_clip_adam<64>(net, a, as_stream(stream));
    DRL_LAUNCH_CHECK("clip_adam_kernel");
    return DRL_OK;
}

}  // extern "C"
