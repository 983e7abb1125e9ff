// rollout256.cu -- fused rollout (deep_rl/ppo.py:110-141) for the 256-wide actor-critic.
// One CTA = 128 environments for all T steps; the ACTOR's W2 (128 KB bf16) stays in shared memory.  Per step:
//   S0   owner threads (one per env, float64 state in registers): observation -> obs[t] in HBM and the [obs_hi|1|obs_lo]
//        operand tile; layer 1 is the same K = 16 GEMM as in the update (identical operands => identical z1)
//   P0   all 512 compute threads: h1 = tanh(z1) -> four bf16 K-chunks; the layer-2 GEMM (M128 N256 K256) is issued chunk by
//        chunk behind them
//   P1   h2 = tanh(z2 + b2), partial head sums (64 units per thread), exchange among the four threads of a row
//   S3   owners: logits, Philox inverse-CDF sample, log-prob, fp64 env step with auto-reset and episode statistics, stores
// The actor phases (S0's operand tile, P0, P1, the logits sum and the issuer's MMAs) live in drl_h256.cuh, shared with
// evaluate256_kernel (eval256.cu), so that an evaluation computes the same logits as the rollout bit for bit.
// The critic is not needed to advance the environments: values V(obs[t]) for all (T+1) x N stored observations are computed
// afterwards by one batched forward pass of the critic (mlp256_kernel in forward mode, update256.cu) -- a plain GEMM-shaped
// launch instead of a second 128 KB weight image per step.
#include "drl_env.cuh"
#include "drl_h256.cuh"
#include "drl_tc_common.cuh"

namespace drl {

int check_env(const drl_env_t* env);
drl_ep_log_t log_or_empty(const drl_ep_log_t* log);

namespace h256 {

int launch_forward256(const drl_net_t* net, const float* packed, const float* obs, int64_t n, float* logits, float* value,
                      int only_net, cudaStream_t st);

template <int KIND>
__global__ void __launch_bounds__(TC_THREADS, 1) rollout256_kernel(drl_env_t env, const float* __restrict__ packed, int T, uint64_t step0,
                                                                   drl_rollout_buf_t buf, drl_ep_log_t log,
                                                                   const drl_ctrl_t* __restrict__ ctrl) {
    if (ctrl != nullptr) step0 = ctrl->env_step;
    using SP = EnvSpec<KIND>;
    constexpr int O = SP::O, A = SP::A, OP = SP::OP;
    using P = Packed256<O, A>;
    using S = RoSmem256<O, A>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* tW2 = sm + S::OFF_W2;
    unsigned char* tACT = sm + S::OFF_ACT;
    unsigned char* tW1B = sm + S::OFF_W1B;
    const float* sB2 = reinterpret_cast<const float*>(sm + S::OFF_B2);
    const float* sW4 = reinterpret_cast<const float*>(sm + S::OFF_W4);
    const float* sB4 = reinterpret_cast<const float*>(sm + S::OFF_B4);
    unsigned char* tOBS = sm + S::OFF_OBS;
    float* xch = reinterpret_cast<float*>(sm + S::OFF_XCH);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + S::OFF_BAR);   // 0 weights, 1 layer 1, 2 layer 2
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
        bulk_g2s(sm + S::OFF_B2, packed + P::B2, HH * 4, bars);
        bulk_g2s(sm + S::OFF_W4, packed + P::W4, A * HH * 4, bars);
        bulk_g2s(sm + S::OFF_B4, packed + P::B4, 16u, bars);
    }
    const uint32_t tmem = *slot;
    mbar_wait(bars, 0);

    if (is_mma_warp) {
        const uint32_t aW2 = smem_u32(tW2), aACT = smem_u32(tACT), aW1B = smem_u32(tW1B), aOBS = smem_u32(tOBS);
        for (int t = 0; t < T; ++t) actor_issue_step(tmem, aOBS, aW1B, aACT, aW2, bars);
        umma::fence_before_sync();
        __syncthreads();
        umma::tmem_dealloc(tmem, 512);
        return;
    }

    const int q = warp & 3, j = warp >> 2;
    const int r = q * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
    const bool owner_warp = j == 0;
    const int N = env.num_envs;
    const int n = blockIdx.x * TC_TILE + r;
    const bool own = owner_warp && n < N;
    const uint32_t gid = env.env_gid0 + (uint32_t)n;
    const uint32_t off0 = umma::sw128_off(r, 2 * j), off1 = umma::sw128_off(r, 2 * j + 1);

    EnvLane e;
    e.s[0] = e.s[1] = e.s[2] = e.s[3] = 0.0; e.elapsed = 0; e.ep_ret = 0.0f; e.ep_len = 0;
    if (own) env_load(e, env, n);

    for (int t = 0; t <= T; ++t) {
        // ---- S0: observation of the current state -> HBM; for t < T also the layer-1 operand tile ----
        if (owner_warp) {
            float obs[OP];
#pragma unroll
            for (int i = 0; i < OP; ++i) obs[i] = 0.0f;
            if (own) {
                env_observation<KIND>(e.s, obs);
                float4* o4 = reinterpret_cast<float4*>(buf.obs + ((size_t)t * N + n) * OP);
#pragma unroll
                for (int qq = 0; qq < OP / 4; ++qq) o4[qq] = make_float4(obs[4 * qq], obs[4 * qq + 1], obs[4 * qq + 2], obs[4 * qq + 3]);
            }
            if (t < T) actor_l1_row<O, OP>(tOBS, r, obs);
        }
        if (t == T) break;            // the last observation needs no action (its value comes from the critic pass)
        umma::fence_before_sync();
        named_bar_arrive(RB_L1, RB_ALL);

        // ---- P0: h1 chunks ----
        actor_h1_chunks(trow, tACT, off0, off1, j, bars, (uint32_t)t & 1u);

        // ---- P1: layer-2 epilogue and partial head sums ----
        actor_head_partials<A>(trow, sB2, sW4, xch, j, r, bars, (uint32_t)t & 1u);
        umma::fence_before_sync();
        named_bar_sync(RB_QUAD + q, 128);

        // ---- S3: owners: sample, env step ----
        if (own) {
            const size_t i0 = (size_t)t * N + n;
            float l[A];
            actor_logits<A>(xch, sB4, r, l);
            if (buf.logits != nullptr) {
#pragma unroll
                for (int a = 0; a < A; ++a) buf.logits[i0 * A + a] = l[a];
            }
            const uint64_t step = step0 + (uint64_t)t;
            const uint4 rr = philox_seeded(env.seed, gid, (uint32_t)step, (uint32_t)(step >> 32), TAG_ACTION);
            float lp;
            const int act = sample_categorical<A>(l, u01_f32(rr.x), lp);
            buf.act[i0] = (uint8_t)act;
            buf.logp[i0] = lp;
            float reward;
            const bool done = env_step<KIND>(e, act, reward, env.seed, gid, step, env.max_episode_steps, log);
            buf.rew[i0 + N] = reward;
            buf.done[i0 + N] = done ? 1 : 0;
        }
        named_bar_sync(RB_QUAD + q, 128);      // the exchange buffer is rewritten in the next step
    }
    if (own) env_store(e, env, n);
    umma::fence_before_sync();
    __syncthreads();
}

template <int KIND>
static int launch_rollout256_kind(const drl_env_t& env, const drl_net_t* net, const float* packed, int T, uint64_t step0,
                                  const drl_rollout_buf_t& buf, const drl_ep_log_t& log, cudaStream_t st, const drl_ctrl_t* ctrl) {
    using SP = EnvSpec<KIND>;
    const int smem = RoSmem256<SP::O, SP::A>::TOTAL;
    DRL_CUDA(cudaFuncSetAttribute(rollout256_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int blocks = (env.num_envs + TC_TILE - 1) / TC_TILE;
    rollout256_kernel<KIND><<<blocks, TC_THREADS, smem, st>>>(env, packed, T, step0, buf, log, ctrl);
    DRL_LAUNCH_CHECK("rollout256_kernel");
    // values of every stored observation, V(obs[t]) for t = 0..T: one batched forward pass of the critic
    return launch_forward256(net, packed, buf.obs, (int64_t)(T + 1) * env.num_envs, nullptr, buf.val, 1, st);
}

int launch_rollout256(const drl_env_t& env, const drl_net_t* net, const float* packed, int T, uint64_t step0, const drl_rollout_buf_t& buf,
                      const drl_ep_log_t& log, cudaStream_t st, const drl_ctrl_t* ctrl) {
    if (env.kind == DRL_ENV_CARTPOLE) return launch_rollout256_kind<DRL_ENV_CARTPOLE>(env, net, packed, T, step0, buf, log, st, ctrl);
    if (env.kind == DRL_ENV_MOUNTAINCAR) return launch_rollout256_kind<DRL_ENV_MOUNTAINCAR>(env, net, packed, T, step0, buf, log, st, ctrl);
    return launch_rollout256_kind<DRL_ENV_ACROBOT>(env, net, packed, T, step0, buf, log, st, ctrl);
}

}  // namespace h256
}  // namespace drl
