// reinforce_ops.cu -- REINFORCE on the device-resident CartPole (SURVEY.md 8f-2; deep_rl/reinforce.py:38-77).
//   policy   nn.Sequential(Linear(4, 128), Dropout(p = 0.6), ReLU, Linear(128, 2), Softmax)          reinforce.py:38-44
//   episode  probs = agent(obs); a ~ Categorical(probs); log_prob; env.step until done               reinforce.py:55-67
//   returns  returns[:step] += gamma ** flip(arange(step)) * reward  = discounted reward-to-go       reinforce.py:67
//            -> drl_gae with lambda = 1 and a zero value plane (the reverse-time scan kernel, gae_ops.cu)
//   loss     b_returns = (R - mean) / (std + exp(-5)); policy_loss = sum(-log_prob * b_returns)       reinforce.py:71-74
//   step     Adam(lr = 1e-2), no clipping                                                            reinforce.py:45,75-77
// One warp per environment, lane l owns hidden units 4l .. 4l+3; N environments run one episode each per iteration (the
// reference runs them one after the other; N = 1 is the reference's schedule).  Env physics, TimeLimit and the episode log are the
// PPO path's (drl_env.cuh); the dropout mask of (env, step) is 128 Philox uniforms (one block per lane, TAG_DROPOUT), regenerated
// in the backward pass instead of being stored.
#include "drl_env.cuh"
#include "drl_update.cuh"

namespace drl {

int check_env(const drl_env_t* env);
drl_ep_log_t log_or_empty(const drl_ep_log_t* log);

constexpr int RH = 128;                 // hidden width
constexpr int RP = 4 * RH + RH + 2 * RH + 2;      // 898 parameters: 0.weight [128][4], 0.bias [128], 3.weight [2][128], 3.bias [2]
constexpr int RPP = (RP + 3) / 4 * 4;   // row stride of the per-episode gradient scratch (16-byte aligned rows)
constexpr uint32_t TAG_DROPOUT = 4;
constexpr float KEEP = 0.4f, DSCALE = 2.5f;        // Dropout(p = 0.6): keep with probability 0.4, scale by 1 / 0.4

struct LaneWeights {
    float w1[4][4], b1[4], w2[2][4];
};
__device__ __forceinline__ void load_lane_weights(LaneWeights& w, const float* __restrict__ p, int lane) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float4 r = *reinterpret_cast<const float4*>(p + (4 * lane + j) * 4);
        w.w1[j][0] = r.x; w.w1[j][1] = r.y; w.w1[j][2] = r.z; w.w1[j][3] = r.w;
        w.b1[j] = p[4 * RH + 4 * lane + j];
        w.w2[0][j] = p[5 * RH + 4 * lane + j];
        w.w2[1][j] = p[6 * RH + 4 * lane + j];
    }
}

// keep flags of this lane's four units for (env gid, step): caller-provided bits (teacher forcing) or the Philox draw
__device__ __forceinline__ uint32_t dropout_keep4(const uint32_t* __restrict__ mask_bits, size_t step_env, uint64_t seed, uint32_t gid,
                                                  uint64_t step, int lane) {
    if (mask_bits != nullptr) return (mask_bits[step_env * 4 + (lane >> 3)] >> (4 * (lane & 7))) & 0xFu;
    const uint4 r = philox_seeded(seed, gid, (uint32_t)step, ((uint32_t)(step >> 32) & 0xFFFFu) | ((uint32_t)lane << 16), TAG_DROPOUT);
    return (u01_f32(r.x) < KEEP ? 1u : 0u) | (u01_f32(r.y) < KEEP ? 2u : 0u) | (u01_f32(r.z) < KEEP ? 4u : 0u) | (u01_f32(r.w) < KEEP ? 8u : 0u);
}

// forward of one observation: z (pre-activation), h (after dropout + ReLU) for the lane's units, logits for the warp
__device__ __forceinline__ void policy_forward(const LaneWeights& w, const float (&x)[4], uint32_t keep, float b2_0, float b2_1,
                                               float (&z)[4], float (&h)[4], float (&logit)[2]) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        z[j] = fmaf(x[3], w.w1[j][3], fmaf(x[2], w.w1[j][2], fmaf(x[1], w.w1[j][1], fmaf(x[0], w.w1[j][0], w.b1[j]))));
        const float d = ((keep >> j) & 1u) ? z[j] * DSCALE : 0.0f;      // Dropout, then ReLU (reinforce.py:40-41)
        h[j] = d > 0.0f ? d : 0.0f;
        s0 = fmaf(h[j], w.w2[0][j], s0);
        s1 = fmaf(h[j], w.w2[1][j], s1);
    }
    logit[0] = warp_sum(s0) + b2_0;
    logit[1] = warp_sum(s1) + b2_1;
}

// One episode per environment.  Planes are [T+1][N] with the PPO path's one-slot shift (rew[t+1], done[t+1] belong to act[t]);
// steps after the end of an episode are written as reward 0 / done 1, so that the lambda = 1 scan leaves zeros there.
__global__ void __launch_bounds__(128) reinforce_episode_kernel(drl_env_t env, const float* __restrict__ params, int T, uint64_t step0,
                                                                float* __restrict__ obs, uint8_t* __restrict__ act,
                                                                float* __restrict__ rew, uint8_t* __restrict__ done,
                                                                int32_t* __restrict__ ep_len_out, uint32_t* __restrict__ mask_bits_out,
                                                                drl_ep_log_t log) {
    const int lane = threadIdx.x & 31;
    const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int N = env.num_envs;
    if (n >= N) return;
    const uint32_t gid = env.env_gid0 + (uint32_t)n;
    LaneWeights w;
    load_lane_weights(w, params, lane);
    const float b2_0 = params[7 * RH], b2_1 = params[7 * RH + 1];
    EnvLane e;
    e.s[0] = e.s[1] = e.s[2] = e.s[3] = 0.0; e.elapsed = 0; e.ep_ret = 0.0f; e.ep_len = 0;
    if (lane == 0) {      // observation = env.reset() (reinforce.py:55): a fresh draw keyed by the step index before the episode
        env_reset_state<DRL_ENV_CARTPOLE>(e.s, env.seed, gid, step0 - 1);
    }
    bool alive = true;
    int len = 0;
    for (int t = 0; t < T; ++t) {
        float x[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) x[i] = __shfl_sync(0xffffffffu, (float)e.s[i], 0);
        const size_t i0 = (size_t)t * N + n;
        if (lane == 0) *reinterpret_cast<float4*>(obs + i0 * 4) = alive ? make_float4(x[0], x[1], x[2], x[3]) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (!alive) {
            if (lane == 0) { act[i0] = 0; rew[i0 + N] = 0.0f; done[i0 + N] = 1; }
            continue;
        }
        const uint64_t step = step0 + (uint64_t)t;
        const uint32_t keep = dropout_keep4(nullptr, 0, env.seed, gid, step, lane);
        if (mask_bits_out != nullptr) {
            uint32_t word = keep << (4 * (lane & 7));
            word |= __shfl_xor_sync(0xffffffffu, word, 1); word |= __shfl_xor_sync(0xffffffffu, word, 2); word |= __shfl_xor_sync(0xffffffffu, word, 4);
            if ((lane & 7) == 0) mask_bits_out[i0 * 4 + (lane >> 3)] = word;
        }
        float z[4], h[4], logit[2];
        policy_forward(w, x, keep, b2_0, b2_1, z, h, logit);
        int a = 0;
        if (lane == 0) {
            const uint4 rr = philox_seeded(env.seed, gid, (uint32_t)step, (uint32_t)(step >> 32), TAG_ACTION);
            float lp;
            a = sample_categorical<2>(logit, u01_f32(rr.x), lp);
            act[i0] = (uint8_t)a;
            float reward;
            drl_ep_log_t nolog = log;
            // env_step resets the state on done (auto-reset); the episode ends here, the next iteration draws its own start state
            const bool d = env_step<DRL_ENV_CARTPOLE>(e, a, reward, env.seed, gid, step, env.max_episode_steps, nolog);
            rew[i0 + N] = reward;
            done[i0 + N] = d ? 1 : 0;
            alive = !d;
        }
        alive = __shfl_sync(0xffffffffu, alive ? 1 : 0, 0) != 0;
        len += 1;
    }
    if (lane == 0) {
        *reinterpret_cast<float4*>(obs + ((size_t)T * N + n) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        ep_len_out[n] = len;
    }
}

// Per-environment gradient of policy_loss = sum_t -log_prob_t * (R_t - mean) / (std + exp(-5)) over the episode's steps
// (reinforce.py:71-74), closed form: dlogit_a' = -Rhat_t (1[a' = a_t] - p_a'), back through Linear / ReLU / Dropout / Linear.
// returns = the discounted reward-to-go plane of drl_gae(lambda = 1, V = 0).  Output: grad_part [N][RPP] (rows padded to a multiple of 4 floats), loss_part [N].
__global__ void __launch_bounds__(128) reinforce_grad_kernel(const float* __restrict__ params, const float* __restrict__ obs,
                                                             const uint8_t* __restrict__ act, const float* __restrict__ returns,
                                                             const int32_t* __restrict__ ep_len, const uint32_t* __restrict__ mask_bits,
                                                             int N, uint64_t seed, uint32_t gid0, uint64_t step0,
                                                             float* __restrict__ grad_part, float* __restrict__ loss_part) {
    const int lane = threadIdx.x & 31;
    const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (n >= N) return;
    LaneWeights w;
    load_lane_weights(w, params, lane);
    const float b2_0 = params[7 * RH], b2_1 = params[7 * RH + 1];
    const int L = ep_len[n];
    // mean and unbiased std of the episode's returns: torch.mean / torch.std (fp32 results; float64 accumulation here)
    double s = 0.0, ss = 0.0;
    for (int t = lane; t < L; t += 32) {
        const double r = (double)returns[(size_t)t * N + n];
        s += r; ss = fma(r, r, ss);
    }
    s = warp_sum(s); ss = warp_sum(ss);
    const double mean_d = L > 0 ? s / L : 0.0;
    const double var_d = L > 1 ? (ss - s * mean_d) / (L - 1) : 0.0;
    const float mean = (float)mean_d;
    const float denom = (float)sqrt(var_d > 0.0 ? var_d : 0.0) + 0.006737946999085467f;      // + np.exp(LOG_STD_MIN), LOG_STD_MIN = -5
    float gw1[4][4], gb1[4], gw2[2][4], gb2[2] = {0.f, 0.f}, loss = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        gb1[j] = 0.f; gw2[0][j] = 0.f; gw2[1][j] = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) gw1[j][i] = 0.f;
    }
    for (int t = 0; t < L; ++t) {
        const size_t i0 = (size_t)t * N + n;
        const float4 o4 = *reinterpret_cast<const float4*>(obs + i0 * 4);
        const float x[4] = {o4.x, o4.y, o4.z, o4.w};
        const uint32_t keep = dropout_keep4(mask_bits, i0, seed, gid0 + (uint32_t)n, step0 + (uint64_t)t, lane);
        float z[4], h[4], logit[2];
        policy_forward(w, x, keep, b2_0, b2_1, z, h, logit);
        const float m = fmaxf(logit[0], logit[1]);
        const float e0 = expf(logit[0] - m), e1 = expf(logit[1] - m);
        const float inv = 1.0f / (e0 + e1);
        const float p0 = e0 * inv, p1 = e1 * inv;
        const int a = act[i0];
        const float logp = logf(a == 0 ? p0 : p1);
        const float rhat = (returns[i0] - mean) / denom;
        loss = fmaf(-logp, rhat, loss);
        const float d0 = -rhat * ((a == 0 ? 1.0f : 0.0f) - p0), d1 = -rhat * ((a == 1 ? 1.0f : 0.0f) - p1);
        gb2[0] += d0; gb2[1] += d1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            gw2[0][j] = fmaf(d0, h[j], gw2[0][j]);
            gw2[1][j] = fmaf(d1, h[j], gw2[1][j]);
            const float dh = fmaf(d1, w.w2[1][j], d0 * w.w2[0][j]);
            const float dz = (((keep >> j) & 1u) && z[j] > 0.0f) ? dh * DSCALE : 0.0f;
            gb1[j] += dz;
#pragma unroll
            for (int i = 0; i < 4; ++i) gw1[j][i] = fmaf(dz, x[i], gw1[j][i]);
        }
    }
    float* g = grad_part + (size_t)n * RPP;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        *reinterpret_cast<float4*>(g + (4 * lane + j) * 4) = make_float4(gw1[j][0], gw1[j][1], gw1[j][2], gw1[j][3]);
        g[4 * RH + 4 * lane + j] = gb1[j];
        g[5 * RH + 4 * lane + j] = gw2[0][j];
        g[6 * RH + 4 * lane + j] = gw2[1][j];
    }
    if (lane == 0) { g[7 * RH] = gb2[0]; g[7 * RH + 1] = gb2[1]; loss_part[n] = loss; }
}

// fixed-order fold of the N per-episode gradients (and losses): grad_out[p] = scale * sum_n grad_part[n][p]
__global__ void __launch_bounds__(256) reinforce_fold_kernel(const float* __restrict__ grad_part, const float* __restrict__ loss_part, int N,
                                                             float scale, float* __restrict__ grad_out, float* __restrict__ loss_out) {
    __shared__ float sh[8][33];
    const int p = blockIdx.x * 32 + threadIdx.x;
    const bool is_loss = p == RP;
    float a = 0.0f;
    if (p <= RP)
        for (int n = threadIdx.y; n < N; n += 8) a += is_loss ? loss_part[n] : grad_part[(size_t)n * RPP + p];
    sh[threadIdx.y][threadIdx.x] = a;
    __syncthreads();
    if (threadIdx.y == 0 && p <= RP) {
        float t = sh[0][threadIdx.x];
#pragma unroll
        for (int y = 1; y < 8; ++y) t += sh[y][threadIdx.x];
        if (is_loss) { if (loss_out) *loss_out = t * scale; }
        else grad_out[p] = t * scale;
    }
}

// torch.optim.Adam (single-tensor path, no weight decay, no clipping) on a flat parameter vector
__global__ void __launch_bounds__(256) adam_step_kernel(float* __restrict__ params, const float* __restrict__ grad, float* __restrict__ m,
                                                        float* __restrict__ v, int64_t n, float beta2, float om_beta1, float om_beta2,
                                                        float eps, float neg_step_size, float bc2_sqrt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float g = grad[i];
    float mi = m[i], vi = v[i], p = params[i];
    adam_apply(g, mi, vi, p, om_beta1, beta2, om_beta2, eps, neg_step_size, bc2_sqrt);
    m[i] = mi; v[i] = vi; params[i] = p;
}

}  // namespace drl

using namespace drl;

extern "C" {

int drl_reinforce_param_count(void) { return RP; }

int drl_reinforce_episodes(const drl_env_t* env, const float* params, int32_t T, uint64_t step0, float* obs, uint8_t* act, float* rew,
                           uint8_t* done, int32_t* ep_len, uint32_t* mask_bits_out, const drl_ep_log_t* log, void* stream) {
    int rc = check_env(env);
    if (rc != DRL_OK) return rc;
    DRL_REQUIRE(env->kind == DRL_ENV_CARTPOLE, "drl_reinforce_episodes: CartPole-v1 only (reinforce.py:26)");
    DRL_REQUIRE(params && obs && act && rew && done && ep_len, "drl_reinforce_episodes: NULL pointer");
    DRL_REQUIRE(T > 0 && step0 >= 1, "drl_reinforce_episodes: T=%d step0=%llu (step0 >= 1: step0 - 1 keys the reset draw)", T,
                (unsigned long long)step0);
    const drl_ep_log_t l = log_or_empty(log);
    const int blocks = (env->num_envs + 3) / 4;
    reinforce_episode_kernel<<<blocks, 128, 0, as_stream(stream)>>>(*env, params, T, step0, obs, act, rew, done, ep_len, mask_bits_out, l);
    DRL_LAUNCH_CHECK("reinforce_episode_kernel");
    return DRL_OK;
}

int drl_reinforce_grad(const float* params, const float* obs, const uint8_t* act, const float* returns, const int32_t* ep_len,
                       const uint32_t* mask_bits, int32_t N, uint64_t seed, uint32_t env_gid0, uint64_t step0, float grad_scale,
                       float* grad_out, float* loss_out, float* grad_part, float* loss_part, void* stream) {
    DRL_REQUIRE(params && obs && act && returns && ep_len && grad_out && grad_part && loss_part, "drl_reinforce_grad: NULL pointer");
    DRL_REQUIRE(N > 0, "drl_reinforce_grad: N=%d", N);
    cudaStream_t st = as_stream(stream);
    reinforce_grad_kernel<<<(N + 3) / 4, 128, 0, st>>>(params, obs, act, returns, ep_len, mask_bits, N, seed, env_gid0, step0, grad_part, loss_part);
    DRL_LAUNCH_CHECK("reinforce_grad_kernel");
    reinforce_fold_kernel<<<(RP + 1 + 31) / 32, dim3(32, 8), 0, st>>>(grad_part, loss_part, N, grad_scale, grad_out, loss_out);
    DRL_LAUNCH_CHECK("reinforce_fold_kernel");
    return DRL_OK;
}

int drl_adam_step(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step, double lr, double beta1,
                  double beta2, double eps, void* stream) {
    DRL_REQUIRE(params && grad && exp_avg && exp_avg_sq, "drl_adam_step: NULL pointer");
    DRL_REQUIRE(n > 0 && step >= 1, "drl_adam_step: n=%lld step=%lld", (long long)n, (long long)step);
    const AdamScalars s = adam_scalars(step, lr, beta1, beta2);
    adam_step_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(params, grad, exp_avg, exp_avg_sq, n, (float)beta2, (float)(1.0 - beta1),
                                                                              (float)(1.0 - beta2), (float)eps, s.neg_step_size, s.bc2_sqrt);
    DRL_LAUNCH_CHECK("adam_step_kernel");
    return DRL_OK;
}

}  // extern "C"
