// eval_ops.cu -- policy evaluation on fresh episodes: every env plays `episodes_per_env` whole episodes of a frozen policy,
// greedy (argmax) or sampled, in one launch.  The counterpart of CleanRL's eval scripts / SB3's evaluate_policy.
//
// Mapping of rollout_kernel (rollout.cu): a warp owns EPW = TL * SUB envs for the whole launch, the forward weights sit in
// shared memory (staged once by TMA bulk copy), the env state stays in registers in fp64.  An env stops stepping after its
// quota of finished episodes; a warp leaves its loop when all its envs have stopped.  Per env-step nothing goes to HBM but
// the finished-episode log entries (and the optional test trace).
//
// Streams: start state = the Philox reset draw of drl_env_reset (step UINT64_MAX), step t uses the rollout's action draw and
// auto-reset keys with step index t, so a CPU oracle env reset with the evaluation key and stepped t = 0, 1, ... reproduces it.
#include "drl_env.cuh"
#include "drl_mlp.cuh"
#include "drl_pack.cuh"

namespace drl {

int check_env(const drl_env_t* env);
int pick_envs_per_warp(int N);     // rollout.cu: DRL_ROLLOUT_EPW forces the evaluation tile too

constexpr int EV_WARPS = 4;

template <int KIND, int SUB, int TL>
__global__ void __launch_bounds__(EV_WARPS * 32) evaluate_kernel(drl_env_t env, const float* __restrict__ packed, int episodes_per_env,
                                                                 int S, bool greedy, drl_ep_log_t log, drl_eval_trace_t tr) {
    using Sp = EnvSpec<KIND>;
    constexpr int O = Sp::O, A = Sp::A, OP = Sp::OP;
    using P = Packed<O, A>;
    constexpr int EPW = TL * SUB;
    constexpr int WS = SUB * OBS_S + H1_S + SUB * OUT_S;

    extern __shared__ __align__(128) float smem[];
    float* sw = smem;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + P::FWD);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* obs_s = smem + P::FWD + 4 + warp * WS;
    float* h1_s = obs_s + SUB * OBS_S;
    float* out_s = h1_s + H1_S;
    stage_params(sw, packed, P::FWD, bar);

    const int N = env.num_envs;
    const int env0 = (blockIdx.x * EV_WARPS + warp) * EPW;
    if (env0 >= N) return;
    const int n = env0 + lane;
    const bool own = lane < EPW && n < N;
    const uint32_t gid = env.env_gid0 + (uint32_t)n;

    EnvLane e;
    e.s[0] = e.s[1] = e.s[2] = e.s[3] = 0.0; e.elapsed = 0; e.ep_ret = 0.0f; e.ep_len = 0;
    if (own) env_reset_state<KIND>(e.s, env.seed, gid, 0xFFFFFFFFFFFFFFFFull);
    int finished = 0;
    bool live = own;          // still short of its episode quota

    int t = 0;
    for (; t < S; ++t) {
        if (__ballot_sync(0xffffffffu, live) == 0u) break;

        if (lane < EPW) {
            float obs[OP];
#pragma unroll
            for (int i = 0; i < OP; ++i) obs[i] = 0.0f;
            if (own) env_observation<KIND>(e.s, obs);
            float* dst = obs_s + (lane / TL) * OBS_S + (lane % TL);
#pragma unroll
            for (int i = 0; i < O; ++i) dst[i * TL] = obs[i];
            if (live) {
                const size_t i0 = (size_t)t * N + n;
                if (tr.obs != nullptr) {
                    float4* o4 = reinterpret_cast<float4*>(tr.obs + i0 * OP);
#pragma unroll
                    for (int q = 0; q < OP / 4; ++q) o4[q] = make_float4(obs[4 * q], obs[4 * q + 1], obs[4 * q + 2], obs[4 * q + 3]);
                }
                if (tr.state != nullptr) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) tr.state[i0 * 4 + i] = e.s[i];
                }
            }
        }
        __syncwarp();

#pragma unroll
        for (int sub = 0; sub < SUB; ++sub) {
            float h2[TL][UPL];
            mlp_forward_tile<O, A, TL>(sw, obs_s + sub * OBS_S, h1_s, out_s + sub * TL * OUT_W, lane, h2);
        }

        // One branch per step holds every lane that steps: env_after_physics aggregates the log over exactly those lanes.
        if (live) {
            const size_t i0 = (size_t)t * N + n;
            float l[A];
#pragma unroll
            for (int a = 0; a < A; ++a) l[a] = out_s[lane * OUT_W + a];
            if (tr.logits != nullptr) {
#pragma unroll
                for (int a = 0; a < A; ++a) tr.logits[i0 * A + a] = l[a];
            }
            int act;
            if (greedy) {
                act = argmax_first<A>(l);
            } else {
                const uint4 r = philox_seeded(env.seed, gid, (uint32_t)t, 0u, TAG_ACTION);     // t < 2^31: high step word 0
                float lp;
                act = sample_categorical<A>(l, u01_f32(r.x), lp);
            }
            if (tr.act != nullptr) tr.act[i0] = (uint8_t)act;
            float reward;
            if (env_step<KIND>(e, act, reward, env.seed, gid, (uint64_t)t, env.max_episode_steps, log)) {
                if (++finished == episodes_per_env) live = false;
            }
        } else if (own && tr.act != nullptr) {
            tr.act[(size_t)t * N + n] = 0xFFu;
        }
        __syncwarp();
    }
    if (own) {
        if (tr.act != nullptr)
            for (; t < S; ++t) tr.act[(size_t)t * N + n] = 0xFFu;
        env_store(e, env, n);
    }
}

template <int KIND, int SUB, int TL>
int launch_evaluate(const drl_env_t& env, const float* packed, int K, bool greedy, const drl_ep_log_t& log, const drl_eval_trace_t& tr,
                    cudaStream_t st) {
    using S = EnvSpec<KIND>;
    constexpr int WS = SUB * OBS_S + H1_S + SUB * OUT_S;
    const size_t smem = sizeof(float) * (Packed<S::O, S::A>::FWD + 4 + EV_WARPS * WS);
    DRL_CUDA(cudaFuncSetAttribute(evaluate_kernel<KIND, SUB, TL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int epc = TL * SUB * EV_WARPS;
    const int blocks = (env.num_envs + epc - 1) / epc;
    evaluate_kernel<KIND, SUB, TL><<<blocks, EV_WARPS * 32, smem, st>>>(env, packed, K, K * env.max_episode_steps, greedy, log, tr);
    DRL_LAUNCH_CHECK("evaluate_kernel");
    return DRL_OK;
}

template <int KIND>
int dispatch_evaluate(int epw, const drl_env_t& env, const float* packed, int K, bool greedy, const drl_ep_log_t& log,
                      const drl_eval_trace_t& tr, cudaStream_t st) {
    if (epw == 4) return launch_evaluate<KIND, 1, 4>(env, packed, K, greedy, log, tr, st);
    if (epw == 8) return launch_evaluate<KIND, 1, 8>(env, packed, K, greedy, log, tr, st);
    if (epw == 16) return launch_evaluate<KIND, 2, 8>(env, packed, K, greedy, log, tr, st);
    return launch_evaluate<KIND, 4, 8>(env, packed, K, greedy, log, tr, st);
}

}  // namespace drl

using namespace drl;

extern "C" int drl_evaluate(const drl_env_t* env, const drl_net_t* net, const float* packed, int32_t episodes_per_env, uint32_t flags,
                            const drl_ep_log_t* log, const drl_eval_trace_t* trace, void* stream) {
    // every failure is an argument error, reported before any CUDA call
    if (check_env(env) != DRL_OK) return DRL_ERR_ARG;
    if (check_net(net) != DRL_OK) return DRL_ERR_ARG;
    DRL_REQUIRE(net->obs_dim == drl_env_obs_dim(env->kind) && net->num_actions == drl_env_num_actions(env->kind),
                "drl_evaluate: net shape does not match env kind %d", env->kind);
    DRL_REQUIRE(net->hidden == H, "drl_evaluate: hidden=%d (evaluation exists for hidden=%d only)", net->hidden, H);
    DRL_REQUIRE(packed != nullptr, "drl_evaluate: packed is NULL");
    DRL_REQUIRE(episodes_per_env >= 1, "drl_evaluate: episodes_per_env=%d", episodes_per_env);
    DRL_REQUIRE((int64_t)episodes_per_env * env->max_episode_steps <= INT32_MAX,
                "drl_evaluate: episodes_per_env * max_episode_steps = %lld exceeds int32",
                (long long)episodes_per_env * env->max_episode_steps);
    DRL_REQUIRE(log != nullptr && log->count != nullptr && log->entries != nullptr, "drl_evaluate: log (count and entries) is required");
    DRL_REQUIRE((int64_t)log->cap >= (int64_t)env->num_envs * episodes_per_env,
                "drl_evaluate: log cap %u < num_envs * episodes_per_env = %lld", log->cap, (long long)env->num_envs * episodes_per_env);
    DRL_REQUIRE((flags & ~DRL_EVAL_GREEDY) == 0u, "drl_evaluate: unknown flags 0x%x", flags);
    drl_eval_trace_t tr;
    memset(&tr, 0, sizeof(tr));
    if (trace) tr = *trace;
    const bool greedy = (flags & DRL_EVAL_GREEDY) != 0u;
    cudaStream_t st = as_stream(stream);
    const int epw = pick_envs_per_warp(env->num_envs);
    const int K = episodes_per_env;
    if (env->kind == DRL_ENV_CARTPOLE) return dispatch_evaluate<DRL_ENV_CARTPOLE>(epw, *env, packed, K, greedy, *log, tr, st);
    if (env->kind == DRL_ENV_MOUNTAINCAR) return dispatch_evaluate<DRL_ENV_MOUNTAINCAR>(epw, *env, packed, K, greedy, *log, tr, st);
    return dispatch_evaluate<DRL_ENV_ACROBOT>(epw, *env, packed, K, greedy, *log, tr, st);
}
