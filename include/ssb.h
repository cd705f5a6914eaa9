/* include/ssb.h -- C ABI of libssb: the batched, B200-native spark-sched-sim scheduling loop.
 *
 * The reference has no FFI: its hot path sits behind the Gymnasium Env API
 * (spark_sched_sim/spark_sched_sim.py:127 `reset`, :188 `step`) and three plug-in ABCs (Scheduler
 * schedulers/scheduler.py:10-18, DataSampler data_samplers/data_sampler.py:9-23, wrappers).  This
 * header is the boundary a binding of that path would use: one `ssb_env` owns B independent
 * environments on one GPU; every entry point is `extern "C"`, takes plain pointers and sizes,
 * returns an int status (0 = ok) and never throws.  INTEGRATION.md shows the ctypes stub that
 * makes `SparkSchedSimEnv` call these.
 *
 * Conventions
 *   - All device work is enqueued on the caller's stream (`stream` = cudaStream_t as void*,
 *     NULL = default stream).  `*_host` variants take HOST buffers, copy, run and synchronise; they run on a stream
 *     of the handle's own and first wait for everything the stream-taking entry points enqueued before them, so a
 *     host-buffer call never overtakes work still queued on a caller's stream.
 *   - The library owns no device memory: the caller passes one workspace allocation
 *     (`ssb_workspace_bytes` tells how big) -- in Python that is a torch uint8 tensor -- and the
 *     observation views returned by `ssb_get_views` are pointers into it.
 *   - Per-environment semantic errors (the reference's ValueError / AssertionError) are reported in
 *     `ssb_obs_hdr.error`: 1..9 = rejected action or reset (state unchanged, see codes below),
 *     >= 1000 = violated internal invariant (environment frozen until the next reset).
 *   - One handle per GPU; a handle is not thread-safe.
 */
#ifndef SSB_H
#define SSB_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSB_ABI_VERSION 10

/* status codes of the entry points */
enum {
    SSB_OK = 0,
    SSB_E_INVALID = -1, /* bad argument / configuration */
    SSB_E_CUDA = -2,    /* CUDA runtime error (ssb_last_cuda_error) */
    SSB_E_WORKSPACE = -3
};

/* per-environment error codes in ssb_obs_hdr.error (mirror the reference's exceptions) */
enum {
    SSB_ENV_OK = 0,
    SSB_ENV_ACTION_SPACE = 1,    /* spark_sched_sim.py:276-277 ValueError */
    SSB_ENV_STAGE_KEY = 2,       /* :284 KeyError (stage_idx >= number of schedulable stages) */
    SSB_ENV_NOT_SCHEDULABLE = 3, /* :286-287 */
    SSB_ENV_ZERO_EXEC = 4,       /* :291-292 */
    SSB_ENV_TOO_MANY_EXEC = 5,   /* :294-295 */
    SSB_ENV_NO_LIMIT = 6,        /* :137-138 */
    SSB_ENV_SAMPLER = 7,         /* tpch.py:106 uncaught KeyError/ValueError */
    SSB_ENV_TAPE_EXHAUSTED = 8,
    SSB_ENV_DONE = 9,            /* step() after termination */
    SSB_ENV_CAPACITY = 10        /* more jobs/stages than the configured capacity */
};

/* env_cfg of the reference (spark_sched_sim.py:34-57, tpch.py:19-26) + batching/capacity knobs */
typedef struct {
    int32_t num_envs;        /* B */
    int32_t num_executors;   /* env_cfg["num_executors"], 1..128 */
    int32_t job_arrival_cap; /* env_cfg["job_arrival_cap"]; <= 0: none (time limit required) */
    int32_t max_jobs;        /* capacity per env; >= job_arrival_cap.  Without a job cap (time-limited arrivals) an
                                episode that needs more jobs is refused at reset with SSB_ENV_CAPACITY in
                                ssb_obs_hdr.error (never silently clipped); the capacity is carved out of the
                                workspace once, so the remedy is a larger handle: the host layer re-creates it with
                                twice the capacity and repeats the reset (batched_env.reset_host(grow=True), always on
                                in the gym facade), or sizes it up front for Exp-distributed limits
                                (required_job_capacity: geometric tail of the job count). */
    int32_t tape_capacity;   /* f64 durations per env for trace replay (0 = no replay support) */
    int32_t log_capacity;    /* event-log rows per env (0 = no event log) */
    double moving_delay;     /* ms */
    double warmup_delay;     /* ms */
    double job_arrival_rate; /* 1/ms */
    double beta;             /* continuous discount (trainer.beta_discount), 0 = undiscounted */
    int32_t flags;           /* SSB_FLAG_* */
    int32_t history_capacity; /* executor-history rows per env and episode (ssb_get_history); 0 = not recorded */
} ssb_config;

#define SSB_FLAG_DECIMA_OBS 1    /* allocate the Decima observation buffers (ssb_decima_obs) */
#define SSB_FLAG_DECIMA_POLICY 2 /* + weights, scratch and outputs of the Decima policy (implies OBS) */

/* Flattened template bank (host pointers; copied to the device by ssb_create).  Layout: see
 * spark-sched-sim_b200/bank.py, which restates tpch.py:118-206. */
typedef struct {
    int32_t num_templates;
    int32_t num_template_stages; /* TS = stage_base[T] */
    int32_t num_template_edges;  /* edge_base[T] */
    int64_t num_values;
    const int32_t *num_stages;    /* [T]   */
    const int32_t *stage_base;    /* [T+1] */
    const int32_t *edge_base;     /* [T+1] */
    const int32_t *edges;         /* [edges][2] (u, v), row-major adjacency order */
    const int32_t *num_tasks;     /* [TS] */
    const double *rough_duration; /* [TS] */
    const uint64_t *parent_mask;  /* [TS] */
    const uint64_t *child_mask;   /* [TS] */
    const uint8_t *present;       /* [TS][3] */
    const uint32_t *dur_off;      /* [TS][3][8] */
    const uint32_t *dur_cnt;      /* [TS][3][8] */
    const double *dur_values;     /* [num_values] */
} ssb_bank;

/* What step()/reset() return besides the graph, one record per environment (device array [B]). */
typedef struct {
    double reward;     /* step() reward (spark_sched_sim.py:208-209) */
    double wall_time;  /* info["wall_time"] */
    int32_t num_nodes; /* N: rows of dag_batch.nodes */
    int32_t num_edges; /* M */
    int32_t num_active_jobs;       /* Ja = len(exec_supplies) */
    int32_t num_committable_execs; /* obs["num_committable_execs"] */
    int32_t source_job_idx;        /* obs["source_job_idx"] (== Ja if none) */
    int32_t num_schedulable;       /* number of valid stage_idx values */
    int32_t error;                 /* SSB_ENV_* or 1000+line */
    uint8_t terminated;
    uint8_t truncated; /* wall_time >= time limit (wrappers/stochastic_time_limit.py:29-30) */
    uint8_t pending;   /* budgeted step only: next decision not reached yet, observation not rewritten */
    uint8_t was_reset; /* auto-reset only: this ssb_step call re-seeded the env instead of applying its action;
                          the observation is the first one of the new episode (reward 0) */
} ssb_obs_hdr;

/* Device views of the observation slabs (fixed stride per environment). */
typedef struct {
    ssb_obs_hdr *hdr;       /* [B] */
    float *nodes;           /* [B][node_stride][3]: remaining tasks, most recent duration, schedulable */
    int32_t *edge_links;    /* [B][edge_stride][2], relabelled to observation node ids */
    int32_t *dag_ptr;       /* [B][job_stride + 1] */
    int32_t *exec_supplies; /* [B][job_stride] */
    int32_t node_stride, edge_stride, job_stride, pad;
} ssb_views;

/* Counters for measurement (device array [B]); zeroed by ssb_create / ssb_reset_stats. */
typedef struct {
    uint64_t decisions;   /* step() calls accepted */
    uint64_t events;      /* timeline events popped */
    uint64_t sched_scans; /* full schedulability scans (spark_sched_sim.py:505) */
    uint64_t sum_nodes, sum_edges, sum_jobs; /* over emitted observations */
    uint64_t observations;
    uint64_t episodes;    /* completed (terminated or truncated) */
} ssb_stats;

typedef struct ssb_env ssb_env;

int ssb_abi_version(void);
const char *ssb_last_cuda_error(void);

/* bytes of device workspace needed for (cfg, bank) */
int ssb_workspace_bytes(const ssb_config *cfg, const ssb_bank *bank, size_t *bytes);

/* builds a handle over `workspace` (device memory, >= ssb_workspace_bytes, 256-B aligned) on CUDA
 * device `device`; uploads the bank.  Replaces SparkSchedSimEnv.__init__ (spark_sched_sim.py:34). */
int ssb_create(const ssb_config *cfg, const ssb_bank *bank, int device, void *workspace,
               size_t workspace_bytes, ssb_env **out);
int ssb_destroy(ssb_env *env);

/* parity mode: give environment `env_index` a pre-sampled job sequence (+ optional duration tape;
 * tape == NULL keeps the Philox task stream).  HOST pointers.  Takes effect at the next reset. */
int ssb_load_trace(ssb_env *env, int32_t env_index, int32_t n_jobs, const double *t_arrival,
                   const int32_t *tmpl, const double *tape, int64_t n_tape);
int ssb_clear_trace(ssb_env *env, int32_t env_index);

/* reset(seed, options={"time_limit"}) for every env with mask[i] != 0 (mask NULL = all).
 * DEVICE pointers: seeds u64[B], time_limits f64[B] (NULL = +inf), mask u8[B]. */
int ssb_reset(ssb_env *env, const uint64_t *seeds, const double *time_limits, const uint8_t *mask,
              void *stream);
/* step(action) for every env (mask NULL = all).  DEVICE pointers i32[B].
 * max_events <= 0: reference semantics -- every env runs until its next scheduling decision.
 * max_events  > 0: asynchronous-vector-env mode -- each env processes at most that many timeline
 *   events in this call; an env that has not reached its next decision is flagged
 *   ssb_obs_hdr.pending = 1 (observation left as it was) and the next ssb_step call on it ignores
 *   its action and continues.  Results per env are identical to the unbounded call; only the
 *   interleaving across envs changes (no env waits for the batch's longest event chain). */
int ssb_step(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
             int32_t max_events, void *stream);

/* Vector-env auto-reset ("next step" mode): when enabled, an ssb_step call on an env whose episode is over
 * (terminated, or truncated by its time limit) re-seeds it with seed + seed_step * reset_count
 * (rollout_worker.py:118-120, the rule ssb_rollout_fair uses), ignores the action, writes the new episode's
 * first observation and sets ssb_obs_hdr.was_reset -- what a caller's `if done: env.reset(seed=...)` does,
 * without a separate ssb_reset launch per call. */
int ssb_set_autoreset(ssb_env *env, int32_t enable, uint64_t seed_step);

/* StochasticTimeLimit (wrappers/stochastic_time_limit.py:5-31) on the device: with mean_ms > 0 every reset that is
 * not given an explicit time limit -- ssb_reset with time_limits == NULL, and every auto-reset of the step API and
 * of the fused rollouts -- draws the new episode's limit ~ Exp(mean_ms) from the LIMIT stream of the episode's seed
 * (Philox ctr (0, 0, 3, 0); oracle/philox_ref.py:time_limit_draw).  mean_ms == 0 (default): explicit limits only,
 * auto-resets keep the previous limit. */
int ssb_set_mean_time_limit(ssb_env *env, double mean_ms);

/* same with HOST buffers: copies in, runs, copies the B observation headers out, synchronises */
int ssb_reset_host(ssb_env *env, const uint64_t *seeds, const double *time_limits, const uint8_t *mask,
                   ssb_obs_hdr *hdr_out);
int ssb_step_host(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
                  int32_t max_events, ssb_obs_hdr *hdr_out);
/* ssb_step_host that also returns, per env, the action the built-in fair (dynamic_partition = 1) / FIFO scheduler
 * (round_robin.py:14-49) takes on the observation the call leaves behind -- evaluated inside the step kernel,
 * so a caller that follows (or overrides) the heuristic needs one call and one synchronisation per decision.
 * Envs that are pending / finished get (-1, 1).  HOST outputs i32[B] each. */
int ssb_step_fair_host(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
                       int32_t max_events, int32_t dynamic_partition, ssb_obs_hdr *hdr_out, int32_t *next_stage_idx,
                       int32_t *next_num_exec);

/* The observation graphs of all envs for a HOST caller (what reset() / step() return as obs, spark_sched_sim.py:393-399),
 * packed: env b's rows follow env b-1's, no padding.  Call after ssb_reset_host / ssb_step_host on the same handle.
 *   offsets  HOST i32[(B + 1) * 3]: (first node, first edge, first job) of env b; row B = the totals.
 *   nodes f32[total nodes][3], edge_links i32[total edges][2] (ids local to the env's graph), exec_supplies
 *   i32[total jobs], dag_ptr i32[total jobs + B] (env b's num_active_jobs + 1 entries start at offsets[3b+2] + b);
 *   any of the four may be NULL.  *_capacity: rows the caller's arrays can hold (SSB_E_WORKSPACE if too small --
 *   offsets[] is valid then and tells the sizes needed).
 * scratch: DEVICE, ssb_packed_obs_bytes, 256-byte aligned (the library owns no device memory).  Two launches, the
 * D2H of the offsets, and one D2H per array of exactly the packed size; synchronous. */
typedef struct {
    int32_t *offsets;
    float *nodes;
    int32_t *edge_links, *dag_ptr, *exec_supplies;
    int64_t node_capacity, edge_capacity, job_capacity;
} ssb_packed_obs;
int ssb_packed_obs_bytes(ssb_env *env, size_t *bytes);
int ssb_get_obs_host(ssb_env *env, ssb_packed_obs *out, void *scratch, size_t scratch_bytes);

/* fused rollout: every env takes `num_decisions` decisions with the built-in fair (dynamic_partition
 * = 1) or FIFO (= 0) policy (round_robin.py:14-49), which reads the simulator state directly.
 * The intermediate observation graphs are not materialised: when the call returns, the views hold the
 * observation that is live then (header, graph and reward), and the ssb_stats counters count every
 * observation.  Per-decision rewards are available through ssb_rollout_fair_traj.
 * auto_reset != 0: a finished env re-seeds itself with seed + seed_step * reset_count
 * (rollout_worker.py:118-120) and continues; otherwise it idles once done. */
int ssb_rollout_fair(ssb_env *env, int32_t num_decisions, int32_t dynamic_partition, int32_t auto_reset,
                     uint64_t seed_step, void *stream);
/* One stored transition of a rollout: what RolloutBuffer.add keeps per step besides the observation
 * (trainers/rollout_worker.py:18-46): the wall time of the observation the action was taken on, the
 * action, and the reward step() returned for it. */
typedef struct {
    double wall_time;
    double reward;
    int32_t stage_idx, num_exec; /* env-format action (stage_idx == -1: no-op) */
    int32_t flags;               /* 1: step() terminated, 2: truncated, 4: first decision after a reset,
                                    8: no transition -- this call only re-seeded the env (ssb_rollout_decima) */
    float lgprob;                /* log-probability of the action under the policy (0 for the heuristics) */
} ssb_transition;
/* ssb_rollout_fair that also records every transition: traj = DEVICE ssb_transition[B][num_decisions],
 * row d of env b at traj[b * num_decisions + d]; an env that stops early (auto_reset == 0) leaves
 * its remaining rows untouched. */
int ssb_rollout_fair_traj(ssb_env *env, int32_t num_decisions, int32_t dynamic_partition, int32_t auto_reset,
                          uint64_t seed_step, ssb_transition *traj, void *stream);

/* Fixed-duration rollouts that span resets (RolloutWorkerAsync.collect_rollout, trainers/rollout_worker.py:160-206):
 * every env keeps deciding (fair / FIFO policy, auto-reset with seed + seed_step * reset_count) until its accumulated
 * simulated time in this call reaches rollout_duration (ms) or max_decisions rows are written; the rows' wall_time is
 * that accumulated time, flags 1 / 2 mark the steps after which the env was reset.  num_steps (DEVICE i32[B]) and
 * elapsed (DEVICE f64[B], the buffer's closing wall_times entry) may be NULL.  The envs continue where they stopped
 * at the next call. */
int ssb_rollout_fair_async(ssb_env *env, int32_t max_decisions, double rollout_duration, int32_t dynamic_partition,
                           uint64_t seed_step, ssb_transition *traj, int32_t *num_steps, double *elapsed, void *stream);

/* ---- what the trainer derives from the rollout buffers before a policy update
 * (trainers/trainer.py:172-212 _preprocess_rollouts).  Plain functions on DEVICE buffers, no handle:
 * traj = ssb_transition[B][stride], num_steps = i32[B] rows stored per rollout (clamped to stride),
 * final_wall = f64[B] wall time after each rollout's last step. */
/* ReturnsCalculator._calc_discounted_returns (trainers/utils/returns_calculator.py:67-76):
 * R_k = r_k + exp(-beta * 1e-3 * (t_{k+1} - t_k)) * R_{k+1}, R_n = 0 -> returns f64[B][stride] */
int ssb_discounted_returns(const ssb_transition *traj, const int32_t *num_steps, const double *final_wall,
                           int32_t num_rollouts_total, int32_t stride, double beta, double *returns,
                           void *stream);
/* ReturnsCalculator._calc_differential_returns (returns_calculator.py:52-65, :78-89).  The calculator's state is a
 * window of the latest `cap` steps with a positive duration over all rollouts (CircularArray): window = DEVICE
 * f64[2][cap][2], a ping-pong pair, zero-filled before the first call, with *which (HOST int, 0 at first) naming the
 * current half -- the call flips it.  scratch = DEVICE i32[2 * B + 1].  Steps: the new (dt, reward) rows of all
 * rollouts, in rollout order, replace the oldest rows; avg_num_jobs (DEVICE f64[1], output) = -sum(reward) / sum(dt)
 * over the window, rows added in order; R_k = -(-r_k - dt_k * avg_num_jobs) + R_{k+1} -> returns f64[B][stride]. */
int ssb_differential_returns(const ssb_transition *traj, const int32_t *num_steps, const double *final_wall,
                             int32_t num_rollouts_total, int32_t stride, double *window, int32_t cap, int32_t *which,
                             int32_t *scratch, double *avg_num_jobs, double *returns, void *stream);
/* PPO._compute_loss (trainers/ppo.py:104-140): the clip loss of one mini-batch and the adjoint seeds of its backward
 * pass.  All arrays DEVICE.  The per-sample arrays new_lgprob / old_lgprob / entropy (f32) and returns / baselines
 * (f64) are indexed by idx[i] (i32[n], NULL = 0..n-1): advantage = float(returns - baselines), normalised with the
 * batch mean and unbiased std (+1e-8); ratio = exp(new - old); policy_loss = -mean(min(adv * ratio, adv *
 * clamp(ratio, 1 - clip, 1 + clip))); entropy_loss = -mean(entropy); out f32[4] = { policy_loss + entropy_coeff *
 * entropy_loss, policy_loss, entropy_loss, mean((ratio - 1) - log_ratio) }.  grad_lgprob / grad_entropy (f32[n], in
 * batch order, may be NULL) = d loss / d new_lgprob, d loss / d entropy.  scratch = DEVICE f64[640]. */
int ssb_ppo_loss(const float *new_lgprob, const float *old_lgprob, const float *entropy, const double *returns,
                 const double *baselines, const int32_t *idx, int32_t n, float clip_range, float entropy_coeff,
                 double *scratch, float *out, float *grad_lgprob, float *grad_entropy, void *stream);
/* TrainableScheduler.update_parameters (schedulers/scheduler.py:37-54) after the backward pass: clip_grad_norm_(grads,
 * max_grad_norm) (skipped when max_grad_norm <= 0), then one torch.optim.Adam step (no weight decay, no amsgrad) on
 * the flat parameter vector (the ssb_set_decima_weights layout).  All arrays DEVICE f32[n]; step = 1 for the first
 * update; scratch = DEVICE f64[128]; grad_norm_out (DEVICE f32[1], may be NULL) receives the norm before clipping.
 * A non-finite norm (the reference's clip_grad_norm_(error_if_nonfinite=True) raises) leaves param / exp_avg /
 * exp_avg_sq untouched: check grad_norm_out.
 * With several GPUs the caller all-reduces `grad` (NCCL, mean) before this call. */
int ssb_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int32_t n, int32_t step, float lr,
                  float beta1, float beta2, float eps, float max_grad_norm, double *scratch, float *grad_norm_out,
                  void *stream);
/* Baseline.average (trainers/utils/baselines.py:12-37): consecutive groups of `group_size` rollouts ran the
 * same job sequence; baseline[b][k] = mean over the group of every member's returns linearly interpolated
 * (np.interp) at rollout b's step time k -> baselines f64[B][stride].  group_size <= 128. */
int ssb_group_baselines(const ssb_transition *traj, const double *returns, const int32_t *num_steps,
                        int32_t num_rollouts_total, int32_t stride, int32_t group_size, double *baselines,
                        void *stream);
/* evaluates the built-in policy on the current observations -> DEVICE i32[B] each */
int ssb_fair_actions(ssb_env *env, int32_t dynamic_partition, int32_t *stage_idx, int32_t *num_exec,
                     void *stream);

/* RandomScheduler.schedule (random_scheduler.py:7-32) on the device, one decision per env with mask[i] != 0
 * (mask NULL = all); DEVICE i32[B] outputs; advances each served env's RANDOM-stream counter.
 * The law is the reference's: a job drawn uniformly among the active jobs that have a schedulable stage, its
 * find_stage choice as stage_idx (-1 when there is none), num_exec uniform on [1, num_committable_execs].  The draws
 * come from the episode seed's Philox RANDOM stream (ctr (decision index in the episode, 0, 5, 0);
 * tests/random_policy_spec.py), not from the reference's RandomState.  Envs that are done, frozen by an
 * error, pending or masked out get (-1, 1) and keep their counter. */
int ssb_random_actions(ssb_env *env, const uint8_t *mask, int32_t *stage_idx, int32_t *num_exec, void *stream);
/* fused random-policy rollout: ssb_rollout_fair's contract with the random policy; traj (DEVICE
 * ssb_transition[B][num_decisions], lgprob 0) may be NULL */
int ssb_rollout_random(ssb_env *env, int32_t num_decisions, int32_t auto_reset, uint64_t seed_step,
                       ssb_transition *traj, void *stream);
/* fixed-duration random-policy rollout: ssb_rollout_fair_async's contract with the random policy; traj (DEVICE
 * ssb_transition[B][max_decisions], lgprob 0), num_steps and elapsed may be NULL.  A draw depends only on the episode
 * seed and the decision's index in the episode, so the same seeds give the same actions as ssb_rollout_random. */
int ssb_rollout_random_async(ssb_env *env, int32_t max_decisions, double rollout_duration, uint64_t seed_step,
                             ssb_transition *traj, int32_t *num_steps, double *elapsed, void *stream);

int ssb_get_views(ssb_env *env, ssb_views *out);

/* Decima's observation adapter on the device (schedulers/decima/env_wrapper.py:69-143 and
 * make_dag_layer_edge_masks, schedulers/decima/utils.py:238-267), computed from the current state
 * of every env; needs SSB_FLAG_DECIMA_OBS.  Same node/edge/job order as the base observation. */
typedef struct {
    float *features;        /* [B][node_stride][5]: cap/E, +-1 source flag, supply/E, remaining/200,
                               remaining*duration/1e5 (float32 arithmetic as in the reference) */
    uint8_t *stage_mask;    /* [B][node_stride] schedulable flag */
    int32_t *commit_caps;   /* [B][job_stride]: exec_mask[j] = first commit_caps[j] of E entries */
    uint64_t *edge_bits;    /* [B][edge_stride]: bit k set <=> edge in edge_masks[k] */
    int32_t *depth;         /* [B]: number of edge masks (message passing depth) */
    int32_t node_stride, edge_stride, job_stride, pad;
    uint8_t *frontier_mask; /* [B][node_stride] 1 = no incoming edge in the observed graph, i.e. every parent has
                               completed -- the "frontier" of heuristics/utils.py:5-37 (Job.frontier_stages) */
} ssb_decima_views;
int ssb_decima_obs(ssb_env *env, void *stream);
int ssb_get_decima_views(ssb_env *env, ssb_decima_views *out);

/* Decima policy on the device (DecimaScheduler.schedule, schedulers/decima/scheduler.py:71-99):
 * observation adapter -> DAG-GNN encoder -> stage scores -> sample -> executor-count scores ->
 * sample, one decision for every env; needs SSB_FLAG_DECIMA_POLICY and weights.
 *   weights: HOST, 20 802 floats, the tensors of models/decima/model.pt concatenated in
 *            state_dict order (each row-major).
 *   forced_stage / forced_num_exec: DEVICE i32[B] or NULL; an entry >= 0 replaces the sampled index
 *            (replaying recorded actions); sampling uses the Philox DECIMA stream of the env's seed,
 *            ctr (decision index in the episode, policy stream of the env, 4, 0) (ssb_set_policy_streams).
 *   stage_idx_out / num_exec_out: DEVICE i32[B] or NULL, in the ENV's action format
 *            (DecimaActWrapper, env_wrapper.py:33-34: num_exec + 1), ready for ssb_step. */
typedef struct {
    float *stage_logits; /* [B][node_stride]: scores of the schedulable stages, action[3] of them */
    float *exec_logits;  /* [B][exec_stride]: scores of num_exec = 0 .. cap-1 for the chosen job */
    int32_t *action;     /* [B][4]: stage_idx, job_idx, num_exec (Decima format), #stage candidates */
    float *lgprob;       /* [B]: log pi(stage) + log pi(num_exec) */
    int32_t node_stride, exec_stride;
    float *entropy;      /* [B]: (H(stage distribution) + H(num_exec distribution)) / log(E * num_nodes), the
                            per-observation entropy evaluate_actions returns (scheduler.py:131-137, utils.py:26-42) */
} ssb_policy_views;
int ssb_set_decima_weights(ssb_env *env, const float *weights, int32_t n_floats);
int ssb_decima_policy(ssb_env *env, const int32_t *forced_stage, const int32_t *forced_num_exec,
                      int32_t *stage_idx_out, int32_t *num_exec_out, void *stream);
int ssb_get_policy_views(ssb_env *env, ssb_policy_views *out);
/* Per-env policy sampling streams (the reference's rollout workers each own a torch RNG): streams = HOST u32[B],
 * NULL = all 0.  Env b's Decima actions are drawn at Philox ctr (decision index in the episode, streams[b], 4, 0),
 * key = the episode seed, so envs that share a seed (one job sequence, several rollouts) still sample their own
 * actions; stream 0 is the default and gives the draws of a handle that never called this.  The streams belong to
 * the handle, not to the episode: ssb_reset, ssb_reset_host, auto-resets and the resets inside the Decima rollouts
 * keep them.  The random scheduler's RANDOM stream (ssb_random_actions) does not use them.  Synchronises the
 * device. */
int ssb_set_policy_streams(ssb_env *env, const uint32_t *streams);
/* One of the policy's seven MLPs (make_mlp, schedulers/decima/utils.py:45-64) applied to caller-provided rows on the
 * tensor-core path the policy uses: mlp = 0 mlp_prep (5 -> 16), 1 mlp_msg, 2 mlp_update (16 -> 16), 3 DagEncoder
 * (21 -> 16), 4 GlobalEncoder (16 -> 16), 5 stage score head (53 -> 1), 6 executor-count score head (36 -> 1), in
 * state_dict order.  x = DEVICE f32[n_rows][in], out = DEVICE f32[n_rows][out].  A building block for callers that
 * assemble their own inputs, and the accuracy probe of the tests (against an fp64 evaluation). */
int ssb_decima_mlp_rows(ssb_env *env, int32_t mlp, const float *x, int32_t n_rows, float *out, void *stream);
/* Rows the last ssb_decima_policy / ssb_decima_evaluate call pushed through each of the policy's MLPs, for
 * measurement (HOST int64[8], synchronous): [0] nodes (mlp_prep and the DagEncoder each see every node), [1] sink
 * nodes (mlp_update, scheduler.py:207-211), [2] schedulable stages (stage score head), [3] active jobs
 * (GlobalEncoder), [4] executor-count rows, [5] message senders and [6] receivers summed over the levels
 * (mlp_msg / mlp_update, :214-232), [7] the multiply-adds of those MLPs at the model's real widths (App. E). */
int ssb_decima_work(ssb_env *env, int64_t *out);
/* Stored observations and their re-evaluation -- RolloutBuffer.obsns (rollout_worker.py:18-46) and
 * DecimaScheduler.evaluate_actions (scheduler.py:101-139), forward pass only:
 *   ssb_decima_snapshot: runs the adapter and copies what the policy reads of every env's observation (header,
 *     edge list, dag_ptr, the adapter's features / masks / caps / level bits / depth) into dst (DEVICE,
 *     ssb_decima_snapshot_bytes).
 *   ssb_decima_evaluate: evaluates the policy on a stored snapshot with the given actions (DEVICE i32[B] each, in
 *     Decima's format: stage_idx = index among the schedulable stages, num_exec in [0, cap)) and writes
 *     lgprob_out / entropy_out (DEVICE f32[B], may be NULL).  The envs' state, current observation and sampling
 *     stream are left untouched. */
int ssb_decima_snapshot_bytes(ssb_env *env, size_t *bytes);
int ssb_decima_snapshot(ssb_env *env, void *dst, void *stream);
int ssb_decima_evaluate(ssb_env *env, const void *snapshot, const int32_t *stage_sel, const int32_t *exec_sel,
                        float *lgprob_out, float *entropy_out, void *stream);
/* Mini-batches drawn over ALL stored samples of an iteration (trainers/ppo.py:52-70: RolloutDataset +
 * DataLoader(shuffle=True)): builds in dst (DEVICE, ssb_decima_snapshot_bytes) a snapshot whose slot i holds the
 * stored observation of sample (step src_step[i], environment src_env[i]) out of `snapshots` (DEVICE: num_steps
 * consecutive blocks of ssb_decima_snapshot_bytes, block k = the ssb_decima_snapshot taken at step k).  src_step /
 * src_env: DEVICE i32[B]; src_step[i] < 0 leaves slot i empty (an observation that takes no part in ssb_decima_evaluate
 * / ssb_decima_backward).  dst is then used like any snapshot (ssb_decima_snapshot_load, ssb_decima_evaluate). */
int ssb_decima_snapshot_gather(ssb_env *env, const void *snapshots, int32_t num_steps, const int32_t *src_step,
                               const int32_t *src_env, void *dst, void *stream);
/* For the policy update, where forward and backward pass of one mini-batch work on the same stored observation:
 * ssb_decima_snapshot_load parks the live observation and puts the stored one in place, ssb_decima_evaluate with
 * snapshot == NULL evaluates it, ssb_decima_backward differentiates that evaluation, ssb_decima_snapshot_unload
 * restores the live observation.  No step / reset / policy call on the handle between load and unload. */
int ssb_decima_snapshot_load(ssb_env *env, const void *snapshot, void *stream);
int ssb_decima_snapshot_unload(ssb_env *env, void *stream);
/* The backward pass of evaluate_actions (loss.backward(), schedulers/scheduler.py:42) for the observation / actions
 * of the last ssb_decima_evaluate / ssb_decima_policy call: loss seeds -> score heads (ssb_decima_head_adjoint,
 * ssb_decima_head_backward) -> global summary (GlobalEncoder, scheduler.py:260-276) -> job summaries (DagEncoder,
 * :244-257) -> with through_node_encoder != 0 also NodeEncoder (:173-241: the message-passing levels in reverse,
 * sinks, mlp_prep).  grad_weights (DEVICE f32[20 802], the ssb_set_decima_weights layout) is accumulated into;
 * with through_node_encoder == 0 NodeEncoder's tensors (mlp_prep / mlp_msg / mlp_update) are left untouched and
 * grad_node_embeddings (DEVICE f32[B][node_stride][16], overwritten) = d loss / d NodeEncoder's output; with
 * through_node_encoder != 0 that buffer is working storage.  The policy's intermediate buffers (embeddings,
 * messages) are overwritten: run ssb_decima_evaluate again before anything that reads them.
 * The message-passing levels are replayed once, their input rows saved in the scratch (room for three rows per node
 * slot; longer level lists fall back to recomputing the levels per level); the call synchronises the stream once
 * (it reads the lists' lengths).
 * scratch: DEVICE, ssb_decima_backward_bytes, 16-byte aligned. */
int ssb_decima_backward_bytes(ssb_env *env, size_t *bytes);
/* Attaches (NULL: detaches) the scratch the coming ssb_decima_backward calls will be given.  While attached,
 * ssb_decima_evaluate stores every message-passing level's input rows into it as a by-product of its forward pass
 * (the tile kernels write the rows they gathered), and an ssb_decima_backward with this scratch that follows such an
 * evaluation skips its own replay of the levels.  (List-driven policy modes; the fused small-batch kernel and any
 * other policy call in between fall back to the replay.) */
int ssb_decima_attach_backward_scratch(ssb_env *env, void *scratch);
int ssb_decima_backward(ssb_env *env, const float *grad_lgprob, const float *grad_entropy, float *grad_weights,
                        float *grad_node_embeddings, int32_t through_node_encoder, void *scratch, void *stream);
/* First stage of the backward pass of evaluate_actions -- the adjoint of utils.evaluate (decima/utils.py:26-42:
 * softmax, clamp_probs, log-prob of the stored action, entropy) and of the aggregation scheduler.py:131-137: from
 * grad_lgprob / grad_entropy (DEVICE f32[B]: d loss / d lgprob, d loss / d entropy of every env, e.g. ssb_ppo_loss's
 * adjoint seeds) to d loss / d scores of the stage head (grad_stage_logits, DEVICE f32[B][node_stride]) and of the
 * executor-count head (grad_exec_logits, DEVICE f32[B][exec_stride]); strides as in ssb_policy_views, zeros outside
 * the candidates.  Uses the scores and actions of the last ssb_decima_evaluate / ssb_decima_policy call. */
int ssb_decima_head_adjoint(ssb_env *env, const float *grad_lgprob, const float *grad_entropy,
                            float *grad_stage_logits, float *grad_exec_logits, void *stream);
/* Second stage: backward of the two score heads' MLPs (StagePolicyNetwork / ExecPolicyNetwork,
 * scheduler.py:279-385) for the candidates of the last ssb_decima_evaluate / ssb_decima_policy call.
 * grad_weights (DEVICE f32[20 802], the ssb_set_decima_weights layout) is ACCUMULATED into (zero it first).
 * grad_stage_inputs (DEVICE f32[num stage candidates][56], may be NULL) / grad_exec_inputs (DEVICE
 * f32[num executor-count rows][40], may be NULL) receive d loss / d input row in list order (stage rows: node
 * features 5, node embedding 16, job embedding 16, global embedding 16, padding; executor-count rows: 3 job
 * features, job embedding 16, global embedding 16, count / E, padding); stage_inputs / exec_inputs (same shapes, may
 * be NULL) the gathered input rows themselves.  num_rows (HOST int32[2], may be NULL) = the two row counts; the
 * call synchronises the stream when it is given. */
int ssb_decima_head_backward(ssb_env *env, const float *grad_stage_logits, const float *grad_exec_logits,
                             float *grad_weights, float *grad_stage_inputs, float *grad_exec_inputs,
                             float *stage_inputs, float *exec_inputs, int32_t *num_rows, void *stream);
/* Decima rollout collection (trainers/rollout_worker.py:135-157 with DecimaScheduler): num_decisions times
 * { ssb_decima_policy (sampled actions) ; ssb_step(max_events) } for every env, everything stream-ordered on the
 * device, each call's (wall time, action, lgprob, reward, flags) stored at traj[b * num_decisions + d] (DEVICE,
 * may be NULL).  Finished envs follow ssb_set_autoreset: with it, the call after the end of an episode
 * re-seeds the env (row flagged 8); without it they idle (rows flagged with error SSB_ENV_DONE semantics). */
int ssb_rollout_decima(ssb_env *env, int32_t num_decisions, int32_t max_events, ssb_transition *traj, void *stream);
/* Fixed-duration Decima rollouts that span resets (RolloutWorkerAsync.collect_rollout, trainers/rollout_worker.py:160-206
 * with DecimaScheduler; the reference trains Decima with these when `rollout_duration` is configured): every env keeps
 * deciding with the sampled Decima policy until its accumulated simulated time in this call reaches rollout_duration
 * (ms) or max_decisions rows are written.  Row d of env b at traj[b * max_decisions + d] (DEVICE): wall_time = the
 * accumulated time before the step, action in the env's format, lgprob, reward, flags 1 / 2 = the step ended the
 * episode (the env is then re-seeded with seed + seed_step * reset_count before its next decision, which carries
 * flag 4).  num_steps (DEVICE i32[B]) / elapsed (DEVICE f64[B], the buffer's closing wall_times entry) may be NULL.
 * Envs that have reached their duration take no part in the remaining rounds (no policy rows, no step, sampling stream
 * untouched) and continue where they stopped at the next call.  Synchronises the stream every few rounds. */
int ssb_rollout_decima_async(ssb_env *env, int32_t max_decisions, double rollout_duration, uint64_t seed_step,
                             ssb_transition *traj, int32_t *num_steps, double *elapsed, void *stream);
/* The stored observations of the two Decima rollouts (RolloutBuffer.obsns, rollout_worker.py:18-46): while a store
 * is attached, every transition row (b, d) that ssb_rollout_decima (d = decision index of the call) or
 * ssb_rollout_decima_async (d = env b's row) writes also stores env b's observation -- the one its action was sampled
 * on -- in slot b of block d of `snapshots` (DEVICE: capacity consecutive blocks in the ssb_decima_snapshot format,
 * ssb_decima_snapshot_bytes each; ssb_decima_snapshot_gather reads them), and the Decima-format action at
 * stage_sel[d][b] / exec_sel[d][b] (DEVICE i32[capacity][B]).  Rows without a transition (re-seed only, a finished
 * env idling, an env past its duration) write nothing; only the rows in use of each part are written.  The rollouts
 * refuse (SSB_E_INVALID) num_decisions / max_decisions > capacity.  snapshots == NULL detaches.  Refused while a
 * snapshot is loaded (ssb_decima_snapshot_load) and on a handle without the policy. */
int ssb_decima_attach_rollout_store(ssb_env *env, void *snapshots, int32_t capacity, int32_t *stage_sel,
                                    int32_t *exec_sel);
/* Episode statistics that survive resets (RecordEpisodeStatistics for the batched env, and the reference's
 * job_duration_buff, spark_sched_sim.py:83, :243-245, :697).  The caller owns the memory, all DEVICE:
 *   episodes      ssb_episode[B][capacity]: a ring of finished episodes per env, or NULL with capacity 0
 *   job_durations f64[B][window]: a ring of completed-job durations (ms) per env, or NULL with window 0
 *   cursors       ssb_episode_cursor[B]; NULL detaches (nothing is written from then on)
 * What is recorded:
 *   - One record per episode, for the step whose observation first reports terminated or truncated
 *     (wall_time >= time_limit, the test of the observation header), written by the call that ran that step (before
 *     any reset that follows it): ssb_step (eager and budgeted), the *_host steps, the fused fair / FIFO / random
 *     rollouts (sync and async) and the Decima rollouts.  Env b's record k goes to
 *     episodes[b][k % capacity]; cursors[b].episodes counts the records.  A truncated env that is stepped again writes
 *     no second record.  No record is written for an episode abandoned by an explicit ssb_reset / ssb_reset_host, an
 *     env frozen by an invariant error (ssb_obs_hdr.error >= 1000), or a reset refused with SSB_ENV_CAPACITY /
 *     SSB_ENV_NO_LIMIT.  An episode that is live when the log is attached counts its decisions from the attach.
 *   - job_time and sum_job_duration are summed serially in job-index order (f64, no contraction), so a host loop
 *     over the jobs restates them bit for bit.
 *   - Every job completion (spark_sched_sim.py:697 appends it there) puts t_completed - t_arrival at
 *     job_durations[b][n % window], n = cursors[b].jobs_completed before the completion, in completion-time order
 *     (job index among equal times: the order of the facade's host deque, env.py; the reference appends in event
 *     order, so two jobs that complete at the same wall time may stand in the other order than there).  The
 *     window and jobs_completed are brought up to date by every call that steps the envs, before it returns (and
 *     inside the fused rollouts before each in-kernel reset).  Resets do
 *     not touch the window, as in the reference: completions of episodes that were later abandoned count too.
 * Attaching fills the library-use fields of the cursors from the live state (stream-ordered on `stream`) and leaves
 * episodes / jobs_completed as given: zero them for a fresh log, keep them to continue one (e.g. on a re-created
 * handle).  The rings are not read by the library except for ssb_collect_stats [6..7].  ssb_reset_stats keeps the
 * decision count of a live episode right.  Refused (SSB_E_INVALID): capacity or window < 0, a NULL ring with a
 * positive size or a ring with size 0. */
typedef struct {              /* one finished episode, 64 B */
    uint64_t seed;            /* the episode's seed */
    double wall_time;         /* wall time of the observation that ended it (ms) */
    double time_limit;        /* the episode's limit (+inf if none) */
    double job_time;          /* sum over arrived jobs of min(t_completed, wall_time) - t_arrival (job-ms):
                                 metrics.avg_num_jobs * wall_time, and minus the undiscounted episode return when
                                 beta = 0 (up to rounding) */
    double sum_job_duration;  /* sum over completed jobs of t_completed - t_arrival (ms) */
    int32_t decisions;        /* step() calls accepted in the episode (ssb_stats.decisions counting) */
    int32_t jobs_arrived, jobs_completed;
    int32_t flags;            /* 1 terminated, 2 truncated */
    int32_t episode;          /* index of the episode since the env's last ssb_reset (0 = the one ssb_reset started) */
    int32_t pad;
} ssb_episode;
typedef struct {              /* per env, 32 B */
    int64_t episodes;         /* episodes recorded since the counts were zeroed; slot = episodes % capacity */
    int64_t jobs_completed;   /* completions recorded; slot = jobs_completed % window */
    uint64_t decisions0;      /* library use: ssb_stats.decisions at the live episode's start */
    int32_t ended;            /* library use: the live episode has been recorded */
    int32_t logged;           /* library use: completions of the live episode already in the window */
} ssb_episode_cursor;
int ssb_attach_episode_log(ssb_env *env, ssb_episode *episodes, int32_t capacity, double *job_durations,
                           int32_t window, ssb_episode_cursor *cursors, void *stream);
/* collect_stats (trainers/rollout_worker.py:122-129) over all envs as SUMS that can be all-reduced across GPUs:
 * out = DEVICE f64[8]: [0] sum over envs of avg_num_jobs = (total job time so far) / wall_time
 * (metrics.py:15-16; envs at wall_time 0 skipped), [1] number of envs counted in [0], [2] completed jobs,
 * [3] job arrivals (completed + active), [4] sum of the completed jobs' durations in ms (current episodes only),
 * [5] sum of wall times, [6] with an episode log that has a job-duration window: sum over the envs with at least one
 * stored duration of the mean of that env's stored durations (ms) -- the reference's env.avg_job_duration, the mean
 * of its last `window` completions across resets -- and [7] the number of such envs; 0 and 0 otherwise.
 * Fixed summation order (deterministic). */
int ssb_collect_stats(ssb_env *env, double *out, void *stream);
/* device pointer to ssb_stats[B] */
int ssb_get_stats(ssb_env *env, ssb_stats **out);
int ssb_reset_stats(ssb_env *env, void *stream);
/* development aid: device pointer to u64[B][16] per-phase cycle counters; they are only advanced by a
 * library built with -DSSB_PROFILE (profiles/phase_breakdown.py), otherwise they stay zero */
int ssb_get_debug_counters(ssb_env *env, uint64_t **out);

/* results (HOST outputs, synchronous): per-job arrival/completion time, template and state
 * (0 = not arrived yet, 1 = active, 2 = completed) of env_index; any output may be NULL */
int ssb_get_jobs(ssb_env *env, int32_t env_index, int32_t *n_jobs, double *t_arrival,
                 double *t_completed, int32_t *tmpl, uint8_t *state, int32_t capacity);
/* event log rows [lo, hi) of env_index (needs log_capacity > 0); *n_rows = rows logged so far */
int ssb_get_log(ssb_env *env, int32_t env_index, int64_t lo, int64_t hi, int64_t *n_rows, double *t,
                uint8_t *type, int16_t *job, int16_t *stage, int32_t *task, int16_t *exec,
                double *t_accepted);

/* Executor history (components/executor.py:25-44 `history`, Executor.add_history; the renderer's input,
 * spark_sched_sim.py:408-424): every add_history call of env_index's current episode in call order -- t[i] = the
 * wall time of the call (= the release time that closes the executor's previous entry), exec[i] = executor id,
 * job[i] = the job the executor belongs to from then on (-1 = common pool).  Called when an executor arrives at a
 * job (:445) and when an idle executor of a saturated job drains to the common pool (:782).  Executor e's list in
 * the reference's format is [[t_1, -1], [t_2, job_1], ..., [None, job_n]] over its rows (t_k, job_k).  Needs
 * ssb_config.history_capacity > 0; *n_rows = calls so far (may exceed the stored capacity).  HOST outputs,
 * synchronous; any output may be NULL. */
int ssb_get_history(ssb_env *env, int32_t env_index, int64_t *n_rows, double *t, int16_t *exec, int16_t *job,
                    int64_t capacity);

#ifdef __cplusplus
}
#endif
#endif
