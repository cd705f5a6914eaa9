// ssb_rollout.cuh -- the fused heuristic rollouts on top of the simulator (ssb_sim.cuh): the decision loops of the
// fixed-count (rollout_w) and fixed-duration (rollout_async_w) rollouts, templated on the policy so that the fair
// (ssb_api.cu) and random (ssb_random.cu) kernels run the same loops in their own units, and the auto-reset and
// transition-row steps they share with k_step.
#pragma once
#include "ssb_env.cuh"
#include "ssb_sim.cuh"

namespace ssb {

// the caller's `if terminated or truncated: env.reset(seed=...)` (rollout_worker.py:118-120, :150-153):
// seed = base_seed + seed_step * reset_count.  `lane` is the kernel's threadIdx.x & 31 (the same value as sim.lane,
// but reading sim.lane here moves the kernels' code).
__device__ __forceinline__ void auto_reset_w(Sim &sim, int lane, uint64_t seed_step)
{
    const uint64_t seed = sim.h->base_seed + seed_step * (uint64_t)sim.h->reset_count;
    const double tl = sim.next_time_limit(seed);
    const bool was_trunc = !sim.h->done;
    __syncwarp();
    if (lane == 0) { sim.h->reset_count += 1; if (was_trunc) sim.stats->episodes++; }
    sim.reset_w(seed, tl);  // writes its observation in full (or, on a capacity error, a zeroed header): owes nothing
}

// RolloutBuffer.add (rollout_worker.py:34-40) minus the observation, for the decision (a, n) just stepped; `fresh` is 4
// for the first decision after an in-kernel reset.  The heuristics have no log-probability.  Returned rather than
// stored through a row pointer, so that `traj[i] = transition_row(...)` computes the row's address after its fields
// (C++17 sequences the right operand of = first), in the order the kernels' code was measured with.
__device__ __forceinline__ ssb_transition transition_row(const Sim &sim, double wall_time, int a, int n, int fresh)
{
    ssb_transition t;
    t.wall_time = wall_time; t.reward = sim.oh->reward; t.stage_idx = a; t.num_exec = n;
    t.flags = (sim.oh->terminated ? 1 : 0) | (sim.oh->truncated ? 2 : 0) | fresh;
    t.lgprob = 0.0f;
    return t;
}

// The body of a fused rollout kernel for env b: `num_decisions` decisions of `policy(sim, policy_arg, a, n)` in one
// launch, finished episodes re-seeded in the kernel when auto_reset is set, transitions recorded when traj is given.
// Only the observation that is live when the loop ends is read (by the caller, after the launch): the decisions
// write its header and counters, the graph (and the reward, without traj) is left owed and written once at the end.
// (An env left pending by a budgeted ssb_step finishes that step first and ignores the action drawn for it.)
// b and lane come from the kernel: computed here, b would lose the range that the kernel's __launch_bounds__ gives
// threadIdx.x.  The policy's kernel argument (policy_arg) is passed at every decision, not captured by the policy: a
// capture is read once at kernel entry and held across the loop.  Either way the kernels' code moves: k_rollout_fair
// with a capturing lambda ran about 0.5 % slower at C2 (one B200, 1000 W power limit).
template <int NS, class Policy>
__device__ __forceinline__ void rollout_w(const Params &p, int b, int lane, const Policy &policy, int policy_arg,
                                          int num_decisions, int auto_reset, uint64_t seed_step, ssb_transition *traj)
{
    Sim sim(p, b, lane);
#ifdef SSB_PROFILE
    const long long t_start = clock64();
#endif
    int d = 0, fresh = 0;
    while (d < num_decisions) {
        if (sim.h->error) break;
        if (sim.h->done || sim.oh->truncated) {
            if (!auto_reset) break;
            fresh = 4;
            auto_reset_w(sim, lane, seed_step);
            continue;
        }
        int a = -1, n = 1;
#ifdef SSB_PROFILE
        long long tp0 = clock64();
#endif
        policy(sim, policy_arg, a, n);
#ifdef SSB_PROFILE
        if (lane == 0) p.prof[(size_t)b * 16 + 8] += (unsigned long long)(clock64() - tp0);
#endif
        const double wall0 = sim.oh->wall_time;
        sim.template step_w<NS, true>(a, n, 0, traj != nullptr);
        if (traj && lane == 0) traj[(size_t)b * num_decisions + d] = transition_row(sim, wall0, a, n, fresh);
        fresh = 0;
        d++;
    }
    __syncwarp();
    if (sim.h->obs_owed) sim.finish_obs_w();
#ifdef SSB_PROFILE
    if (lane == 0) p.prof[(size_t)b * 16 + 10] += (unsigned long long)(clock64() - t_start);
#endif
}

// RolloutWorkerAsync.collect_rollout (trainers/rollout_worker.py:160-206) for env b with `policy(sim, policy_arg, a, n)`:
// the rollout ends when the env's accumulated simulated time reaches `duration` (or after max_decisions rows), resets
// do not end it, and the time axis of the stored rows is that accumulated time.  The step is the eager one (every
// decision writes its observation in full).  b, lane and policy_arg as in rollout_w, and sim is constructed by the
// kernel too: constructed here from p, k_rollout_fair_async's code moves (24 instructions fewer in <1>, 24 more in <2>).
template <int NS, class Policy>
__device__ __forceinline__ void rollout_async_w(Sim &sim, int b, int lane, const Policy &policy, int policy_arg,
                                                int max_decisions, double duration, uint64_t seed_step,
                                                ssb_transition *traj, int32_t *num_steps, double *elapsed_out)
{
    int d = 0, fresh = 0;
    double elapsed = 0.0;
    while (d < max_decisions && elapsed < duration) {
        if (sim.h->error) break;
        if (sim.h->done || sim.oh->truncated) {  // :196-200, applied when the loop comes back around
            fresh = 4;
            auto_reset_w(sim, lane, seed_step);
            continue;
        }
        int a = -1, n = 1;
        policy(sim, policy_arg, a, n);
        const double wall0 = sim.oh->wall_time;
        sim.template step_w<NS>(a, n);
        // rollout_buffer.add(obs, elapsed_time, action, lgprob, reward) (:191)
        if (traj && lane == 0) traj[(size_t)b * max_decisions + d] = transition_row(sim, elapsed, a, n, fresh);
        elapsed += sim.oh->wall_time - wall0;  // the duration of this step (:194)
        fresh = 0;
        d++;
    }
    if (lane == 0) {
        if (num_steps) num_steps[b] = d;
        if (elapsed_out) elapsed_out[b] = elapsed;
    }
}

}  // namespace ssb
