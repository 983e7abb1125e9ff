// drl_update.cuh -- arguments shared by the two implementations of the minibatch gradient
// (FP32 CUDA-core path in update_ops.cu, tcgen05 tensor-core path in update_tc.cu), and the one definition of the
// optimizer-step arithmetic (partial-gradient fold, loss terms, clip, Adam) that every update path uses.
#pragma once
#include "drl_common.cuh"

namespace drl {

constexpr int DRL_MAX_STEPS_PER_LAUNCH = 8;

struct AdamArgs {
    float* params; const float* grad; float* m; float* v; float* packed; float* norm_out;
    int P;
    float grad_scale, max_norm, beta2, om_beta1, om_beta2, eps, neg_step_size, bc2_sqrt;
};

// Optional in-kernel tail of the tensor-core gradient kernel (single GPU): after a grid-wide barrier the CTAs fold
// the partial gradients slice-wise, clip by the global norm and apply Adam -- the whole minibatch step is one launch.
// The fp32 path's fused fold + clip + Adam (reduce_clip_adam_kernel, update_ops.cu) takes the same arguments.
struct TailArgs {
    int enabled;
    AdamArgs a;
    float* grad_out; float* loss_terms_out;
    double* cta_sumsq;        // [gridDim.x]
    uint32_t* ctr;            // [4] grid barriers 1-3, depart (zero between launches); the fp32 fused step uses [0] and [3]
    // multi-GPU (world > 1): symmetric peer buffers, layout = CommLayout
    int world, rank;
    unsigned char* peer[DRL_MAX_RANKS];
    uint32_t seq;
    int* error_flag;
    // graph-replayable launch (drl_ppo_minibatch_update_ctl): Adam scalars and sequence number come from device memory
    const drl_ctrl_t* ctrl;
    int ordinal;
    // one launch = nsteps consecutive, equally sized minibatches (GradArgs.mb_start + s * mb_count, adv_stats[2s], loss terms
    // row s, optimizer step s): by-value Adam scalars per step (ctrl == nullptr)
    int nsteps;
    float neg_step_size_s[DRL_MAX_STEPS_PER_LAUNCH], bc2_sqrt_s[DRL_MAX_STEPS_PER_LAUNCH];
};

// Symmetric buffer of one rank (push protocol): two generations (seq & 1) of [DRL_MAX_RANKS] gradient copies -- rank s WRITES its
// folded slices into slot s of every rank's buffer -- followed by two generations of arrival flags [DRL_MAX_RANKS][FLAG_CTAS]
// (one flag per source rank and CTA slice, holding the sequence number of the step that wrote the slice).
constexpr int FLAG_CTAS = 160;
struct CommLayout {
    size_t xgrad[2], flags[2], rank_stride, total;
};
__host__ __device__ inline CommLayout comm_layout(int64_t P) {
    CommLayout c;
    const size_t g = ((size_t)P * 4 + 255) / 256 * 256;
    c.rank_stride = g;
    c.xgrad[0] = 0; c.xgrad[1] = (size_t)DRL_MAX_RANKS * g;
    c.flags[0] = 2 * (size_t)DRL_MAX_RANKS * g; c.flags[1] = c.flags[0] + sizeof(uint32_t) * DRL_MAX_RANKS * FLAG_CTAS;
    c.total = c.flags[1] + sizeof(uint32_t) * DRL_MAX_RANKS * FLAG_CTAS;
    return c;
}

struct GradArgs {
    const float* packed;
    const float* rec;
    const uint32_t* idx;
    uint32_t mb_start, mb_count;
    const float* adv_stats;   // [2] mean, std
    float clip_coef, ent_coef, vf_coef;
    float* grad_part;         // [gridDim.x][ppad]
    float* loss_part;         // [gridDim.x][LOSS_TERMS]
    int ppad;
    long long* dbg;           // optional cycle stamps (diagnostics), else nullptr
    TailArgs tail;
};

// ---- the optimizer-step arithmetic every update path shares.  The library builds with -fmad=false, so an inlined helper
// rounds exactly as the expression written out in place would: keep each operand order. ----

// Adam's step scalars exactly as torch.optim.adam._single_tensor_adam computes them (Python floats, fp64), optimizer step `step` >= 1
struct AdamScalars { float neg_step_size, bc2_sqrt; };
inline AdamScalars adam_scalars(int64_t step, double lr, double beta1, double beta2) {
    const double bc1 = 1.0 - pow(beta1, (double)step);
    const double bc2 = 1.0 - pow(beta2, (double)step);
    return {(float)(-(lr / bc1)), (float)sqrt(bc2)};
}

// torch.optim.Adam's element update (no weight decay) of one parameter w with state m, v; gsc is the gradient as Adam sees it,
// already scaled and clipped
__device__ __forceinline__ void adam_apply(float gsc, float& m, float& v, float& w, float om_beta1, float beta2, float om_beta2,
                                           float eps, float neg_step_size, float bc2_sqrt) {
    m = m + om_beta1 * (gsc - m);                     // exp_avg.lerp_(grad, 1 - beta1)
    v = v * beta2 + (om_beta2 * gsc) * gsc;           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) / bc2_sqrt + eps;
    w = w + (neg_step_size * m) / denom;              // param.addcdiv_(exp_avg, denom, value=-step_size)
}

// clip_grad_norm_: the gradient's coefficient from its global squared norm; block 0 reports the norm to a.norm_out
__device__ __forceinline__ float clip_coef(double sumsq, const AdamArgs& a) {
    const float norm = (float)sqrt(sumsq);
    const float c = a.max_norm / (norm + 1e-6f);
    const float coef = c < 1.0f ? c : 1.0f;
    if (blockIdx.x == 0 && a.norm_out != nullptr) *a.norm_out = norm;
    return coef;
}

// The LOSS_TERMS row of a minibatch from the five loss sums over its samples {pg, v, entropy, approx_kl, clipped}:
// {loss, pg_loss, v_loss, entropy, approx_kl, clipfrac, 0, 0}
__device__ __forceinline__ void store_loss_terms(float* out, const float* sums, uint32_t mb_count, float ent_coef, float vf_coef) {
    const float inv = 1.0f / (float)mb_count;
    const float pg = sums[0] * inv, vl = 0.5f * sums[1] * inv, en = sums[2] * inv;
    out[0] = pg - ent_coef * en + vl * vf_coef;
    out[1] = pg; out[2] = vl; out[3] = en;
    out[4] = sums[3] * inv; out[5] = sums[4] * inv;
    out[6] = 0.0f; out[7] = 0.0f;
}

// Fixed-order fold of parameter p over the partial rows row0, row0 + 8 stride, ... (< nrows) of one of 8 slices: four
// interleaved accumulators over groups of four rows while a whole group fits, the remaining rows one by one into the first.
// The 8 slice sums are then added in slice order by the caller.
__device__ __forceinline__ float fold_partials(const float* __restrict__ part, int ppad, int p, int row0, int stride, int nrows) {
    const int step = 8 * stride;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int c = row0;
    for (; c + 3 * step < nrows; c += 4 * step) {
        const float v0 = __ldcg(part + (size_t)c * ppad + p);
        const float v1 = __ldcg(part + (size_t)(c + step) * ppad + p);
        const float v2 = __ldcg(part + (size_t)(c + 2 * step) * ppad + p);
        const float v3 = __ldcg(part + (size_t)(c + 3 * step) * ppad + p);
        a0 += v0; a1 += v1; a2 += v2; a3 += v3;
    }
    for (; c < nrows; c += step) a0 += __ldcg(part + (size_t)c * ppad + p);
    return (a0 + a1) + (a2 + a3);
}

// fixed-order fold of `nrows` per-CTA partial gradients / loss sums (update_ops.cu).  Parameters below `critic0` are folded
// over rows 0, stride, 2 stride, ..., the others over rows 1, 1 + stride, ...: stride 1 with critic0 = P folds every row
// (H = 64), stride 2 with critic0 = the actor's parameter count folds the actor over the even rows and the critic over the odd
// ones (H = 256, update256.cu)
int launch_grad_reduce(const GradArgs& g, int nrows, int P, int stride, int critic0, float* grad_out, float* loss_terms_out,
                       cudaStream_t st);

// tensor-core implementation (update_tc.cu)
// grid_out != nullptr: skip the fold of the partials and report the number of partials instead
int launch_grad_tc(const drl_net_t* net, const GradArgs& g, int P, float* grad_out, float* loss_terms_out, cudaStream_t st,
                   int* grid_out = nullptr);
// tensor-core gradient + in-kernel fold / clip / Adam tail (g.tail filled by the caller), one cooperative launch
int launch_grad_tc_fused(const drl_net_t* net, GradArgs& g, cudaStream_t st);

}  // namespace drl
