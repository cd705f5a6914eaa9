// ssb_types.cuh -- device-side state layout of the batched scheduling simulator (libssb).
//
// One environment = one episode of the reference's SparkSchedSimEnv (spark_sched_sim.py:29).
// State is env-major in HBM: every array below is [B][stride] so that the warp that owns an
// environment reads its jobs / stages / executors with consecutive lanes on consecutive records
// (16-byte vector loads for StageRec).  Python objects of the reference collapse as follows:
//   EventQueue (event.py:19)      -> one pending-event slot per executor (every executor has at
//                                    most one TASK_FINISHED/EXECUTOR_READY in flight) + a cursor
//                                    over the pre-sampled, time-ordered job arrivals
//   Job/Stage DAG (job.py, stage.py) -> u64 bitmasks per job (active, frontier, saturated,
//                                    schedulable, selected) + 16-byte counters per stage; the DAG
//                                    itself (parent/child masks) stays in the shared template bank
//   ExecutorTracker pools (executor_tracker.py:38-42) -> CPython-set look-alike tables (u8 slots),
//                                    because set iteration/pop order decides which executor moves
//   _commitments dict-of-dicts    -> one insertion-ordered record list per environment
#pragma once
#include <stdint.h>

#include "../../include/ssb.h"

namespace ssb {

enum : int { EV_JOB_ARRIVAL = 0, EV_TASK_FINISHED = 1, EV_EXECUTOR_READY = 2 };
enum : int { POOL_NONE = 0, POOL_COMMON = 1 };  // job j -> 2 + j, stage node v -> 2 + Jc + v
enum : int { JOB_PENDING = 0, JOB_ACTIVE = 1, JOB_COMPLETED = 2 };

struct __align__(16) StageRec {  // stage.py:8-18 + tracker counters keyed by the stage's pool
    uint16_t remaining;          // num_remaining_tasks
    uint16_t completed;          // num_completed_tasks
    uint16_t num_tasks;
    int16_t job;
    uint8_t commit_to;    // _num_commitments_to_stage
    uint8_t moving_to;    // _num_moving_to_stage
    uint8_t commit_from;  // _num_commitments_from[(job, stage)]
    uint8_t pad;
    float mrd;  // most_recent_duration as the observation sees it (float32)
};
static_assert(sizeof(StageRec) == 16, "StageRec must be one 128-bit load");

struct __align__(16) ExecRec {  // executor.py:4-20 + its pending timeline event
    double ev_t;                // event key (t, seq), event.py:34-35
    double t_acc;               // task.t_accepted (event log only)
    uint32_t ev_seq;
    int32_t ev_task;
    int16_t ev_job, ev_stage;
    int16_t job_id;      // executor.job_id, -1 = None
    int16_t task_stage;  // executor.task.stage_id
    int32_t loc;         // _executor_locations: pool id, POOL_NONE while moving
    uint8_t ev_kind;     // 0 = no pending event, else EV_*
    uint8_t is_executing;
    uint8_t has_task;  // executor.task is not None
    uint8_t pad0;
    int32_t pad1[2];
};
static_assert(sizeof(ExecRec) == 48, "ExecRec layout");

struct __align__(16) JobRec {  // job.py:12-40 + tracker counters keyed by the job
    double t_arrival, t_completed;
    uint64_t active;    // incomplete stages (active_stages)
    uint64_t frontier;  // frontier_stages
    uint64_t sat;       // stages with executor demand <= 0 (spark_sched_sim.py:580-582)
    uint64_t sched;     // this job's slice of self.schedulable_stages
    uint64_t selected;  // this job's slice of self.selected_stages
    int32_t tmpl, node_base, edge_base, ts_base;
    int16_t n_stages;
    int16_t n_local;      // len(local_executors)
    int16_t supply;       // _total_executor_count[job]
    int16_t commit_from;  // _num_commitments_from[(job, None)]
    uint8_t sat_count;    // saturated_stage_count
    uint8_t state;
    int16_t n_obs_edges;  // template edges with both ends in `active`: the job's edges in the observation
    uint8_t logged;       // the episode log's window holds this job's duration (set by Sim::log_job_durations_w)
    uint8_t pad[3];
};
static_assert(sizeof(JobRec) == 96, "JobRec layout");

struct Commit {  // one (src pool -> dst pool: n) entry; list order == dict insertion order
    int32_t src, dst, n;
};

struct PoolHdr {  // PySetObject: mask, fill, used, finger (Objects/setobject.c)
    uint16_t mask, fill, used, finger;
};

struct __align__(16) LogRow {
    double t, t_acc;
    int32_t task;
    int16_t job, stage, exec;
    uint8_t type, pad;
    int32_t pad1;
};
static_assert(sizeof(LogRow) == 32, "LogRow layout");

struct __align__(16) HistRow {  // one Executor.add_history call (executor.py:34-44)
    double t;     // wall time of the call = release time of the executor's previous history entry
    int16_t exec;
    int16_t job;  // job the executor now belongs to, -1 = common pool
    int32_t pad;
};
static_assert(sizeof(HistRow) == 16, "HistRow layout");

struct __align__(16) EnvHdr {
    double wall_time, time_limit, wall_old;
    uint64_t seed, base_seed;
    int64_t log_n;
    uint32_t launch_idx, seq;
    int32_t n_jobs, next_arrival, n_active, n_completed;
    int32_t source, n_sched, n_commits, n_old_active;
    int32_t commit_from_common, commit_to_common, total_none, error;
    int32_t done, trace_jobs, tape_len, n_nodes_total;
    int32_t n_edges_total, reset_count, use_tape, pending;
    uint32_t policy_draws;  // Philox policy-stream counter (on-device action sampling)
    int32_t hist_n;         // add_history calls of this episode (rows beyond hist_cap are counted, not stored)
    int32_t obs_owed;  // k_rollout_fair: parts of the live observation still to be written (Sim::OWE_*), 0 outside it
    // nodes and edges of the observation (active stages of the active jobs, edges between them), kept current where
    // a job's `active` or the active-job list changes, so that the per-decision observation header needs no count pass
    int32_t n_obs_nodes, n_obs_edges;
};
static_assert(sizeof(EnvHdr) == 160, "EnvHdr layout");

// The buffers of ssb_attach_episode_log (caller-owned device memory)
struct EpisodeLog {
    ssb_episode *rec;         // [B][cap] ring of finished episodes (nullptr when cap == 0)
    double *win;              // [B][window] ring of completed-job durations (nullptr when window == 0)
    ssb_episode_cursor *cur;  // [B]
    int32_t cap, window;
};

// Everything a kernel needs, passed by value.
struct Params {
    int B, E, Jc, Sc, Mc, TAB, RT, P, Cc, max_stages;
    int tape_cap, log_cap, job_arrival_cap, hist_cap;
    double moving_delay, warmup_delay, mean_interarrival, beta;
    double mean_time_limit;  // > 0: every reset without an explicit limit draws one (StochasticTimeLimit)
    // template bank (read-only)
    const int32_t *b_num_stages, *b_stage_base, *b_edge_base, *b_num_tasks;
    const int16_t *b_edges;  // [edges][2]
    const double *b_rough;
    const uint64_t *b_parent, *b_child;
    const uint8_t *b_present;  // [TS][4] (3 used)
    const uint2 *b_dur;        // [TS][3][8] (offset, count)
    const double *b_vals;
    const short4 *iv;  // [E+1] executor intervals (tpch.py:237-262): left/right level, left/right level index
    // state
    EnvHdr *hdr;
    ExecRec *exec;     // [B][E]
    JobRec *job;       // [B][Jc]
    StageRec *stage;   // [B][Sc]
    int16_t *active;   // [B][Jc]  active_job_ids
    int16_t *old_act;  // [B][Jc]
    int16_t *reward_ord;  // [B][Jc] job ids in the reward's summation order
    Commit *commits;   // [B][Cc]
    PoolHdr *pool_hdr; // [B][P]
    uint8_t *pool_tab; // [B][P][TAB]
    uint8_t *scr_tab;  // [B][3][TAB]  copy / idle / resize scratch
    uint16_t *rset;    // [B][2][RT]   reward job-id set + resize scratch
    double *trace_t;   // [B][Jc]
    int32_t *trace_tmpl;  // [B][Jc]
    double *tape;      // [B][tape_cap]
    LogRow *log;       // [B][log_cap]
    HistRow *hist;     // [B][hist_cap] executor history (only with ssb_config.history_capacity > 0)
    ssb_stats *stats;  // [B]
    double *stats_part;  // [128][8] partial sums of ssb_collect_stats, then the episode log's descriptor (episode_log)
    unsigned long long *prof;  // [B][16] cycle counters per phase (written only when built with -DSSB_PROFILE)
    // observation slabs
    ssb_obs_hdr *obs_hdr;
    float *obs_nodes;
    int32_t *obs_edges, *obs_dag_ptr, *obs_supplies;
    // Decima observation adapter outputs (nullptr unless SSB_FLAG_DECIMA_OBS)
    float *dec_feat;          // [B][Sc][5]
    uint8_t *dec_stage_mask;  // [B][Sc]
    uint8_t *dec_frontier_mask;  // [B][Sc]
    int32_t *dec_caps;        // [B][Jc]
    uint64_t *dec_edge_bits;  // [B][Mc]
    int32_t *dec_depth;       // [B]
    // Decima policy (nullptr unless SSB_FLAG_DECIMA_POLICY): weights, scratch, outputs
    float *pol_w;             // [20802] state_dict order
    float *pol_h_init, *pol_h, *pol_msg;  // [B][Sc][16]
    float *pol_h_dag, *pol_g;             // [B][Jc][16]
    float *pol_h_glob;                    // [B][16]
    int32_t *pol_row_start;               // [B][Sc]
    float *pol_stage_logits;              // [B][Sc]
    float *pol_exec_logits;               // [B][Epad]
    int32_t *pol_action;                  // [B][4]
    float *pol_lgprob;                    // [B]
    float *pol_entropy;                   // [B]
    char *pol_snap;                       // scratch: the live observation during ssb_decima_evaluate
    int32_t *pol_act_a, *pol_act_n;       // [B] env-format actions of ssb_rollout_decima
    int32_t *traj_d;                      // row index of the rollout-buffer slab being written
    int Epad;
    // tensor-core policy path (ssb_decima_tc.cuh): row lists built per decision by the planning kernels
    int32_t *pl_all, *pl_sink;                     // [B * Sc] flat node ids (b * Sc + n)
    int32_t *pl_cand, *pl_cand_job, *pl_cand_out;  // [B * Sc] schedulable stages: node, job row, logit slot
    int32_t *pl_jobs;                              // [B * Jc] flat job ids (b * Jc + i)
    int32_t *pl_exec;                              // [B * Epad] rows of the executor-count head
    int32_t *pl_lvl;                               // [lvl_cap] senders / receivers of every level
    int32_t *pl_cnt;                               // counters, offsets, cursors (tc::CNT_*)
    int32_t *pl_ncand;                             // [B]
    unsigned long long *pl_bits;                   // [B * Sc][2] levels at which a node sends / receives
    uint32_t *pol_wblob3;  // per-stage bf16 three-term weight blobs (fz::blob3_offset)
    int32_t *pol_cand_rank;  // [B][Sc] rank of a schedulable node among its env's schedulable nodes (its score's slot)
    int32_t *fz_cursor;      // [4] group cursor of the fused policy kernel
    // optional per-env participation mask of one policy call (nullptr = all): an env with pol_active[b] == 0 is treated
    // like a finished one (no rows, action (-1, 1)) and its sampling stream is not advanced
    const uint8_t *pol_active;
    // fixed-duration Decima rollouts (ssb_rollout_decima_async): per-env accumulators of the current call
    double *as_elapsed, *as_wall0;  // [B]
    int32_t *as_rows;               // [B] rows written so far
    uint8_t *as_kind;               // [B] this round: 0 = not taking part, 1 = decision, 2 = reset
    uint8_t *as_fresh;              // [B] the next row is the first after a reset
    int32_t *as_any;                // [1] envs still taking part
    int lvl_cap;
};

// The partial sums of ssb_collect_stats ([STATS_BLOCKS][8]) and, right after them in the same workspace region, the
// descriptor of the log ssb_attach_episode_log attached (cur == nullptr: none).  Reached through p.stats_part so that
// Params keeps its layout: the simulator kernels copy Params to local memory, and a new field reshuffles that copy and
// the registers of the whole fused rollout kernel.
constexpr int STATS_BLOCKS = 128;
constexpr int STATS_PART_DOUBLES = STATS_BLOCKS * 8;
__host__ __device__ inline EpisodeLog *episode_log(const Params &p)
{
    return reinterpret_cast<EpisodeLog *>(p.stats_part + STATS_PART_DOUBLES);
}

}  // namespace ssb
