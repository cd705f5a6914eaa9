// ssb_random.cu -- the random scheduler (RandomScheduler, schedulers/heuristics/random_scheduler.py:7-32) on the device:
// its side of the C ABI (include/ssb.h), one-decision actions and fused random-policy rollouts (fixed decision count
// and fixed simulated duration).
// A translation unit of its own so that nothing here sits next to the simulator kernels of ssb_api.cu (see
// ssb_env.cuh).
#define SSB_RANDOM_POLICY
#include "ssb_env.cuh"
#include "ssb_rollout.cuh"

using namespace ssb;

namespace {
// one decision per env with mask[b] != 0 (mask null = all); done, error-frozen, pending and masked-out envs get
// (-1, 1) and their RANDOM-stream counter stays where it is
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
k_random_actions(Params p, const uint8_t *mask, int32_t *stage_idx, int32_t *num_exec)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    Sim sim(p, b, lane);
    int a = -1, n = 1;
    if ((!mask || mask[b]) && !sim.h->error && !sim.h->done && !sim.h->pending) sim.random_action_w(a, n);
    if (lane == 0) { stage_idx[b] = a; num_exec[b] = n; }
}

// the fused rollout (ssb_rollout.cuh) with the random policy
template <int NS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, NS == 1 ? SSB_NS1_CTAS : SSB_NS2_CTAS)
k_rollout_random(Params p, int num_decisions, int auto_reset, uint64_t seed_step, ssb_transition *traj)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    rollout_w<NS>(p, b, lane, [](Sim &sim, int, int &a, int &n) { sim.random_action_w(a, n); }, 0, num_decisions,
                  auto_reset, seed_step, traj);
}

// the fixed-duration rollout (ssb_rollout.cuh) with the random policy
template <int NS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, NS == 1 ? SSB_NS1_CTAS : SSB_NS2_CTAS)
k_rollout_random_async(Params p, int max_decisions, double duration, uint64_t seed_step, ssb_transition *traj,
                       int32_t *num_steps, double *elapsed_out)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    Sim sim(p, b, lane);
    rollout_async_w<NS>(sim, b, lane, [](Sim &sim, int, int &a, int &n) { sim.random_action_w(a, n); }, 0,
                        max_decisions, duration, seed_step, traj, num_steps, elapsed_out);
}
}  // namespace

extern "C" {

int ssb_random_actions(ssb_env *env, const uint8_t *mask, int32_t *stage_idx, int32_t *num_exec, void *stream)
{
    if (!env || !stage_idx || !num_exec) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    k_random_actions<<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(env->p, mask, stage_idx, num_exec);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_rollout_random(ssb_env *env, int32_t num_decisions, int32_t auto_reset, uint64_t seed_step,
                       ssb_transition *traj, void *stream)
{
    if (!env || num_decisions < 0) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    if (env->p.E <= 32)
        k_rollout_random<1><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(env->p, num_decisions, auto_reset,
                                                                                        seed_step, traj);
    else
        k_rollout_random<2><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(env->p, num_decisions, auto_reset,
                                                                                        seed_step, traj);
    CUDA_TRY(cudaGetLastError());
    if (const int rc_ = ssb_i_episode_log_launch(env, (cudaStream_t)stream)) return rc_;
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_rollout_random_async(ssb_env *env, int32_t max_decisions, double rollout_duration, uint64_t seed_step,
                             ssb_transition *traj, int32_t *num_steps, double *elapsed, void *stream)
{
    if (!env || max_decisions < 0 || !(rollout_duration > 0.0)) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    if (env->p.E <= 32)
        k_rollout_random_async<1><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(
            env->p, max_decisions, rollout_duration, seed_step, traj, num_steps, elapsed);
    else
        k_rollout_random_async<2><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(
            env->p, max_decisions, rollout_duration, seed_step, traj, num_steps, elapsed);
    CUDA_TRY(cudaGetLastError());
    if (const int rc_ = ssb_i_episode_log_launch(env, (cudaStream_t)stream)) return rc_;
    SSB_MARK(env, stream);
    return SSB_OK;
}

}  // extern "C"
