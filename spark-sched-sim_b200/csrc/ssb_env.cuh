// ssb_env.cuh -- what the translation units of libssb share: the handle, status / ordering macros and the internal
// entry points that cross units.  The simulator kernels (ssb_api.cu) and the Decima policy (ssb_policy.cu) are separate
// units ON PURPOSE: the fused rollout kernel is bound by instruction supply, and what else is instantiated in its unit
// moves its code around -- the policy kernels next to it cost the headline 5 % (16.8 M instead of 17.7 M decisions/s,
// profiles/r02_bench_n1_before_split.json); round 1 saw the same with the backward kernels.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "ssb_types.cuh"

namespace ssb {
extern thread_local char g_cuda_err[256];  // ssb_last_cuda_error()
}

#ifndef SSB_WARPS_PER_CTA
#define SSB_WARPS_PER_CTA 4
#endif
constexpr int WARPS_PER_CTA = SSB_WARPS_PER_CTA;
// resident CTAs per SM that the simulator kernels' __launch_bounds__ ask for (fused rollouts of ssb_api.cu and ssb_random.cu)
#ifndef SSB_NS1_CTAS
#define SSB_NS1_CTAS 7  // resident CTAs per SM of the one-slot kernels: 4096 envs = 1024 CTAs of 4 warps must all be resident
#endif
#ifndef SSB_NS2_CTAS
#define SSB_NS2_CTAS 7  // resident CTAs per SM the two-slot kernels (E > 32) are compiled for: 72 registers (some spilling), but 28 warps
                        // per SM and 8192 envs = 2048 CTAs in exactly two rounds of resident CTAs (A/B in profiles/r02_ns2_occupancy.txt)
#endif

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t e_ = (expr);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            snprintf(ssb::g_cuda_err, sizeof(ssb::g_cuda_err), "%s: %s", #expr, cudaGetErrorString(e_)); \
            return SSB_E_CUDA;                                                           \
        }                                                                                \
    } while (0)

// The stream-taking entry points launch on the handle's device whatever the caller's current device is
// (a stream of another device fails the launch with a plain CUDA error instead of an opaque one later).
#define SSB_ON_DEVICE(env)                                                   \
    do {                                                                     \
        int cur_ = -1;                                                       \
        if (cudaGetDevice(&cur_) != cudaSuccess || cur_ != (env)->device) CUDA_TRY(cudaSetDevice((env)->device)); \
    } while (0)

// Ordering between the caller's streams and the handle's own stream (the *_host entry points): every stream-taking
// entry point marks the end of what it enqueued (SSB_MARK), and a *_host call first makes its own stream wait for
// that mark (host_begin) -- work still queued on the caller's stream is never overtaken by a host-buffer call.
#define SSB_MARK(env, stream)                                                             \
    do {                                                                                  \
        if ((cudaStream_t)(stream) != (env)->own_stream) {                                \
            CUDA_TRY(cudaEventRecord((env)->ev_last, (cudaStream_t)(stream)));            \
            (env)->dirty = 1;                                                             \
        }                                                                                 \
    } while (0)


// ------------------------------------------------------------------------------------ workspace
struct Carver {
    char *base;
    size_t off = 0;
    template <typename T>
    T *take(size_t n)
    {
        off = (off + 255) & ~size_t(255);
        T *ptr = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += n * sizeof(T);
        return ptr;
    }
};

struct Dims {
    int TAB, RT, Sc, Mc, P, Cc, max_stages, max_edges;
};

struct BankDev {
    int32_t *num_stages, *stage_base, *edge_base, *num_tasks;
    int16_t *edges;
    double *rough;
    uint64_t *parent, *child;
    uint8_t *present;
    uint2 *dur;
    double *vals;
    short4 *iv;
};


// How ssb_decima_policy runs: row lists + one launch per MLP pass with the TMEM-resident bf16 three-term tiles (the
// default for large batches), or the whole decision of a group of envs in one persistent kernel (one launch: small
// batches, e.g. the single-env facade).
enum { POLICY_TILES = 0, POLICY_FUSED = 1 };

// The stored-observation buffers ssb_decima_attach_rollout_store hands the Decima rollouts (snap == nullptr: none)
struct RolloutStore {
    char *snap;  // [cap] ssb_decima_snapshot blocks
    int32_t cap;
    int32_t *stage_sel, *exec_sel;  // [cap][B]
    bool operator==(const RolloutStore &o) const
    {
        return snap == o.snap && cap == o.cap && stage_sel == o.stage_sel && exec_sel == o.exec_sel;
    }
};

struct ssb_env {
    ssb_config cfg;
    Dims dims;
    ssb::Params p;
    BankDev bank;
    int device;
    char *ws;
    size_t ws_bytes;
    cudaStream_t own_stream;
    int32_t *st_a, *st_n;  // staging for the *_host entry points
    uint64_t *st_seed;
    double *st_tl;
    uint8_t *st_mask;
    int grid;
    int num_sms;
    int dmax;           // upper bound of the message-passing depth: longest template chain - 1
    // CUDA graph of one ssb_rollout_decima decision and the arguments it was captured with
    cudaEvent_t ev;
    cudaEvent_t ev_last;  // recorded after the latest work enqueued on a caller's stream (see SSB_MARK / host_begin)
    int dirty;            // such work exists since the last *_host call
    cudaGraphExec_t dg_exec;
    ssb_transition *dg_traj;
    int dg_k, dg_events, dg_autoreset, no_graph;
    uint64_t dg_seed_step;
    RolloutStore dg_store;
    int policy_mode;    // POLICY_* below (SSB_DECIMA_MODE overrides the default)
    void *bw_scratch;   // ssb_decima_attach_backward_scratch
    int bw_saved;       // the last policy evaluation left its levels' input rows in bw_scratch
    int fused_group;    // environments per group of the fused policy kernel
    int snap_loaded;    // ssb_decima_snapshot_load: a stored observation is in place, the live one parked
    int auto_reset;     // ssb_set_autoreset
    uint64_t auto_seed_step;
    // Decima policy unit only (ssb_policy.cu): the simulator kernels never see these
    uint32_t *pol_streams;  // [B] policy sampling stream of every env (ssb_set_policy_streams), in the workspace
    RolloutStore store;     // ssb_decima_attach_rollout_store
};

// ---- internal entry points across the units (C linkage like the public ones; not exported through include/ssb.h)
extern "C" {
// ssb_api.cu
int ssb_i_step_launch(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
                      int32_t max_events, int32_t *next_a, int32_t *next_n, int dyn, cudaStream_t s,
                      int force_autoreset, uint64_t force_seed_step);
// ssb_policy.cu
int ssb_i_decima_obs(ssb_env *env, cudaStream_t s);  // the observation adapter kernel
void ssb_i_policy_carve(Carver &cv, const ssb_config &c, const Dims &d, ssb::Params &p, uint32_t **pol_streams);
int ssb_i_policy_init(ssb_env *env);
void ssb_i_drop_decision_graph(ssb_env *env);
}
