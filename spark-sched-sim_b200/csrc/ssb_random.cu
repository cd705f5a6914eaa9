// ssb_random.cu -- the random scheduler (RandomScheduler, schedulers/heuristics/random_scheduler.py:7-32) on the device:
// its side of the C ABI (include/ssb.h), one-decision actions and fused random-policy rollouts.
// A translation unit of its own so that nothing here sits next to the simulator kernels of ssb_api.cu (see
// ssb_env.cuh): k_rollout_random keeps its own copy of k_rollout_fair's decision loop for the same reason.
#define SSB_RANDOM_POLICY
#include "ssb_env.cuh"
#include "ssb_sim.cuh"

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

// k_rollout_fair (ssb_api.cu) with the random policy: `num_decisions` decisions per env in one launch, the
// observation deferred to the end of the loop, in-kernel auto-reset, transitions when traj is given.  (An env left
// pending by a budgeted ssb_step finishes that step first and ignores the action drawn for it, as in k_rollout_fair.)
template <int NS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, NS == 1 ? SSB_NS1_CTAS : SSB_NS2_CTAS)
k_rollout_random(Params p, int num_decisions, int auto_reset, uint64_t seed_step, ssb_transition *traj)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    Sim sim(p, b, lane);
    int d = 0, fresh = 0;
    while (d < num_decisions) {
        if (sim.h->error) break;
        if (sim.h->done || sim.oh->truncated) {
            if (!auto_reset) break;
            fresh = 4;
            // rollout_worker.py:118-120: seed = base_seed + seed_step * reset_count
            const uint64_t seed = sim.h->base_seed + seed_step * (uint64_t)sim.h->reset_count;
            const double tl = sim.next_time_limit(seed);
            const bool was_trunc = !sim.h->done;
            __syncwarp();
            if (lane == 0) { sim.h->reset_count += 1; if (was_trunc) sim.stats->episodes++; }
            sim.reset_w(seed, tl);  // writes its observation in full: owes nothing
            continue;
        }
        int a = -1, n = 1;
        sim.random_action_w(a, n);
        const double wall0 = sim.oh->wall_time;
        sim.template step_w<NS, true>(a, n, 0, traj != nullptr);
        if (traj && lane == 0) {  // RolloutBuffer.add (rollout_worker.py:34-40) minus the observation
            ssb_transition t;
            t.wall_time = wall0; t.reward = sim.oh->reward; t.stage_idx = a; t.num_exec = n;
            t.flags = (sim.oh->terminated ? 1 : 0) | (sim.oh->truncated ? 2 : 0) | fresh;
            t.lgprob = 0.0f;  // RandomScheduler returns no log-probability
            traj[(size_t)b * num_decisions + d] = t;
        }
        fresh = 0;
        d++;
    }
    __syncwarp();
    if (sim.h->obs_owed) sim.finish_obs_w();
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
    SSB_MARK(env, stream);
    return SSB_OK;
}

}  // extern "C"
