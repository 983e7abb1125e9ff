// eval256.cu -- policy evaluation on fresh episodes for the 256-wide actor-critic, on tcgen05 (bf16 operands, fp32
// accumulation): the semantics of drl_evaluate (eval_ops.cu) with the numerics of rollout256_kernel.
//
// Mapping of rollout256_kernel (rollout256.cu): one CTA = 128 envs, the actor's W2 (128 KB SW128 image) resident in shared
// memory, W1B / B2 / W4 / B4 staged once by TMA bulk copy, the env state in fp64 registers of the owner threads (warps 0-3).
// Per step the CTA runs the actor phases of drl_h256.cuh -- the same operands, GEMMs, activations and summation order as the
// rollout -- so the logits of an observation are bit-identical to the rollout's, and a sampled evaluation reproduces what the
// training rollout would have done from the same state.  No rollout planes, no critic pass: per env-step nothing goes to HBM
// but the finished-episode log entries (and the optional test trace).
//
// An env stops stepping after its quota of finished episodes; the CTA leaves its loop when all of its 128 envs have stopped.
#include "drl_env.cuh"
#include "drl_h256.cuh"
#include "drl_tc_common.cuh"

namespace drl {

int check_env(const drl_env_t* env);
int check_net(const drl_net_t* net);

namespace h256 {

template <int KIND>
__global__ void __launch_bounds__(TC_THREADS, 1) evaluate256_kernel(drl_env_t env, const float* __restrict__ packed, int episodes_per_env,
                                                                    int S, bool greedy, drl_ep_log_t log, drl_eval_trace_t tr) {
    using SP = EnvSpec<KIND>;
    constexpr int O = SP::O, A = SP::A, OP = SP::OP;
    using P = Packed256<O, A>;
    using SM = RoSmem256<O, A>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* tW2 = sm + SM::OFF_W2;
    unsigned char* tACT = sm + SM::OFF_ACT;
    unsigned char* tW1B = sm + SM::OFF_W1B;
    const float* sB2 = reinterpret_cast<const float*>(sm + SM::OFF_B2);
    const float* sW4 = reinterpret_cast<const float*>(sm + SM::OFF_W4);
    const float* sB4 = reinterpret_cast<const float*>(sm + SM::OFF_B4);
    unsigned char* tOBS = sm + SM::OFF_OBS;
    float* xch = reinterpret_cast<float*>(sm + SM::OFF_XCH);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + SM::OFF_BAR);   // 0 weights, 1 layer 1, 2 layer 2
    uint32_t* slot = reinterpret_cast<uint32_t*>(bars + 3);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool is_mma_warp = warp == TC_COMPUTE / 32;

    if (tid == 0) {
        mbar_init(bars, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 1);
        mbar_fence_init();
    }
    if (is_mma_warp) umma::tmem_alloc(slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    if (tid == 0) {
        mbar_expect_tx(bars, (uint32_t)(HH * HH * 2 + 2 * HH * 8 * 2 + HH * 4 + A * HH * 4 + 16));
        const char* w2 = reinterpret_cast<const char*>(packed + P::W2);
        for (uint32_t off = 0; off < (uint32_t)(HH * HH * 2); off += 32768u) bulk_g2s(tW2 + off, w2 + off, 32768u, bars);
        bulk_g2s(tW1B, packed + P::W1B, 2 * HH * 8 * 2, bars);
        bulk_g2s(sm + SM::OFF_B2, packed + P::B2, HH * 4, bars);
        bulk_g2s(sm + SM::OFF_W4, packed + P::W4, A * HH * 4, bars);
        bulk_g2s(sm + SM::OFF_B4, packed + P::B4, 16u, bars);
    }
    const uint32_t tmem = *slot;
    mbar_wait(bars, 0);

    const uint32_t aW2 = smem_u32(tW2), aACT = smem_u32(tACT), aW1B = smem_u32(tW1B), aOBS = smem_u32(tOBS);
    const int q = warp & 3, j = warp >> 2;
    const int r = q * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
    const bool owner_warp = j == 0;            // warps 0-3; the issuer warp has j = 4
    const int N = env.num_envs;
    const int n = blockIdx.x * TC_TILE + r;
    const bool own = owner_warp && n < N;
    const uint32_t gid = env.env_gid0 + (uint32_t)n;
    const uint32_t off0 = umma::sw128_off(r, 2 * j), off1 = umma::sw128_off(r, 2 * j + 1);

    EnvLane e;
    e.s[0] = e.s[1] = e.s[2] = e.s[3] = 0.0; e.elapsed = 0; e.ep_ret = 0.0f; e.ep_len = 0;
    if (own) env_reset_state<KIND>(e.s, env.seed, gid, 0xFFFFFFFFFFFFFFFFull);
    int finished = 0;
    bool live = own;          // still short of its episode quota; only owner threads of real envs (n < N) are ever live

    // Exit protocol.  The step loop is entered and left by all TC_THREADS threads together: at the top of every step, before
    // anyone touches a named barrier or an mbarrier of that step, every thread (the issuer warp included) takes part in ONE
    // CTA-wide vote, __syncthreads_or(live), and all of them break on its single result.  So every thread runs exactly the same
    // number of steps: the issuer syncs RB_L1 / RB_H1 + c and commits bars[1] / bars[2] exactly once per step that the compute
    // warps run, each compute thread arrives at those barriers and waits on the mbarrier phases (t & 1) of exactly those
    // steps, and each row quarter meets twice at RB_QUAD + q per step -- no thread can wait on a barrier or a phase that others
    // skip.  Envs that stopped (and padding rows n >= N) still have their GEMM rows computed; the results are ignored.  The
    // loop is also bounded by S = K * max_episode_steps, which TimeLimit guarantees to be enough for every quota.  After the
    // loop all threads reach the same trailing fence / __syncthreads / tmem_dealloc sequence.
    int t = 0;
    for (; t < S; ++t) {
        if (__syncthreads_or(live ? 1 : 0) == 0) break;

        if (is_mma_warp) {
            actor_issue_step(tmem, aOBS, aW1B, aACT, aW2, bars);
            continue;
        }

        // ---- S0: observation of the current state -> the layer-1 operand tile (and the trace) ----
        if (owner_warp) {
            float obs[OP];
#pragma unroll
            for (int i = 0; i < OP; ++i) obs[i] = 0.0f;
            if (own) env_observation<KIND>(e.s, obs);
            if (live) {
                const size_t i0 = (size_t)t * N + n;
                if (tr.obs != nullptr) {
                    float4* o4 = reinterpret_cast<float4*>(tr.obs + i0 * OP);
#pragma unroll
                    for (int qq = 0; qq < OP / 4; ++qq) o4[qq] = make_float4(obs[4 * qq], obs[4 * qq + 1], obs[4 * qq + 2], obs[4 * qq + 3]);
                }
                if (tr.state != nullptr) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) tr.state[i0 * 4 + i] = e.s[i];
                }
            }
            actor_l1_row<O, OP>(tOBS, r, obs);
        }
        umma::fence_before_sync();
        named_bar_arrive(RB_L1, RB_ALL);

        // ---- P0: h1 chunks; P1: layer-2 epilogue and partial head sums ----
        actor_h1_chunks(trow, tACT, off0, off1, j, bars, (uint32_t)t & 1u);
        actor_head_partials<A>(trow, sB2, sW4, xch, j, r, bars, (uint32_t)t & 1u);
        umma::fence_before_sync();
        named_bar_sync(RB_QUAD + q, 128);

        // ---- S3: live owners: logits, action, env step.  One branch holds every lane that steps: env_after_physics
        // aggregates the log over exactly those lanes. ----
        if (live) {
            const size_t i0 = (size_t)t * N + n;
            float l[A];
            actor_logits<A>(xch, sB4, r, l);
            if (tr.logits != nullptr) {
#pragma unroll
                for (int a = 0; a < A; ++a) tr.logits[i0 * A + a] = l[a];
            }
            int act;
            if (greedy) {
                act = argmax_first<A>(l);
            } else {
                const uint4 rr = philox_seeded(env.seed, gid, (uint32_t)t, 0u, TAG_ACTION);     // t < 2^31: high step word 0
                float lp;
                act = sample_categorical<A>(l, u01_f32(rr.x), lp);
            }
            if (tr.act != nullptr) tr.act[i0] = (uint8_t)act;
            float reward;
            if (env_step<KIND>(e, act, reward, env.seed, gid, (uint64_t)t, env.max_episode_steps, log)) {
                if (++finished == episodes_per_env) live = false;
            }
        } else if (own && tr.act != nullptr) {
            tr.act[(size_t)t * N + n] = 0xFFu;
        }
        named_bar_sync(RB_QUAD + q, 128);      // the exchange buffer is rewritten in the next step
    }
    if (own) {
        if (tr.act != nullptr)
            for (; t < S; ++t) tr.act[(size_t)t * N + n] = 0xFFu;
        env_store(e, env, n);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (is_mma_warp) umma::tmem_dealloc(tmem, 512);
}

template <int KIND>
static int launch_evaluate256(const drl_env_t& env, const float* packed, int K, bool greedy, const drl_ep_log_t& log,
                              const drl_eval_trace_t& tr, cudaStream_t st) {
    using SP = EnvSpec<KIND>;
    const int smem = RoSmem256<SP::O, SP::A>::TOTAL;
    DRL_CUDA(cudaFuncSetAttribute(evaluate256_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int blocks = (env.num_envs + TC_TILE - 1) / TC_TILE;
    evaluate256_kernel<KIND><<<blocks, TC_THREADS, smem, st>>>(env, packed, K, K * env.max_episode_steps, greedy, log, tr);
    DRL_LAUNCH_CHECK("evaluate256_kernel");
    return DRL_OK;
}

}  // namespace h256
}  // namespace drl

using namespace drl;

extern "C" int drl_evaluate_tc(const drl_env_t* env, const drl_net_t* net, const float* packed, int32_t episodes_per_env, uint32_t flags,
                               const drl_ep_log_t* log, const drl_eval_trace_t* trace, void* stream) {
    // every failure is an argument error, reported before any CUDA call
    if (check_env(env) != DRL_OK) return DRL_ERR_ARG;
    DRL_REQUIRE(net != nullptr, "drl_evaluate_tc: net is NULL");
    if (net->hidden == H) {
        set_error("drl_evaluate_tc: hidden=%d has no tensor-core evaluation; use drl_evaluate", net->hidden);
        return DRL_ERR_UNSUPPORTED;
    }
    DRL_REQUIRE(net->hidden == h256::HH, "drl_evaluate_tc: hidden=%d (tensor-core evaluation exists for hidden=%d only)", net->hidden,
                h256::HH);
    if (check_net(net) != DRL_OK) return DRL_ERR_ARG;
    DRL_REQUIRE(net->obs_dim == drl_env_obs_dim(env->kind) && net->num_actions == drl_env_num_actions(env->kind),
                "drl_evaluate_tc: net shape does not match env kind %d", env->kind);
    DRL_REQUIRE(packed != nullptr, "drl_evaluate_tc: packed is NULL");
    DRL_REQUIRE(episodes_per_env >= 1, "drl_evaluate_tc: episodes_per_env=%d", episodes_per_env);
    DRL_REQUIRE((int64_t)episodes_per_env * env->max_episode_steps <= INT32_MAX,
                "drl_evaluate_tc: episodes_per_env * max_episode_steps = %lld exceeds int32",
                (long long)episodes_per_env * env->max_episode_steps);
    DRL_REQUIRE(log != nullptr && log->count != nullptr && log->entries != nullptr, "drl_evaluate_tc: log (count and entries) is required");
    DRL_REQUIRE((int64_t)log->cap >= (int64_t)env->num_envs * episodes_per_env,
                "drl_evaluate_tc: log cap %u < num_envs * episodes_per_env = %lld", log->cap, (long long)env->num_envs * episodes_per_env);
    DRL_REQUIRE((flags & ~DRL_EVAL_GREEDY) == 0u, "drl_evaluate_tc: unknown flags 0x%x", flags);
    drl_eval_trace_t tr;
    memset(&tr, 0, sizeof(tr));
    if (trace) tr = *trace;
    const bool greedy = (flags & DRL_EVAL_GREEDY) != 0u;
    cudaStream_t st = as_stream(stream);
    const int K = episodes_per_env;
    if (env->kind == DRL_ENV_CARTPOLE) return h256::launch_evaluate256<DRL_ENV_CARTPOLE>(*env, packed, K, greedy, *log, tr, st);
    if (env->kind == DRL_ENV_MOUNTAINCAR) return h256::launch_evaluate256<DRL_ENV_MOUNTAINCAR>(*env, packed, K, greedy, *log, tr, st);
    return h256::launch_evaluate256<DRL_ENV_ACROBOT>(*env, packed, K, greedy, *log, tr, st);
}
