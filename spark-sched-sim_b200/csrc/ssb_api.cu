// ssb_api.cu -- kernels and the C ABI of libssb (include/ssb.h).
//
// Launch geometry of the simulator kernels: one warp per environment, 4 environments per 128-thread CTA,
// grid = ceil(B/4).  At B = 4096 that is 1024 CTAs (~7 per SM on 148 SMs), all resident at once (the one-slot
// kernels are held to 72 registers for that); the kernels are dependency chains per environment bound by
// instruction supply (DESIGN.md 5), so residency is what keeps the SM busy.  The Decima policy is a sequence
// of list-driven tile kernels over all environments (ssb_decima_tc.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>
#include "ssb_env.cuh"
#include "ssb_rollout.cuh"

using namespace ssb;

namespace ssb {
thread_local char g_cuda_err[256] = "";  // ssb_last_cuda_error(); also written by ssb_learn.cu and ssb_policy.cu
}

namespace {
// ------------------------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
k_reset(Params p, const uint64_t *seeds, const double *time_limits, const uint8_t *mask)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    if (mask && !mask[b]) return;
    Sim sim(p, b, lane);
    const uint64_t seed = seeds ? seeds[b] : 0ull;
    if (lane == 0) { sim.h->base_seed = seed; sim.h->reset_count = 1; }
    sim.reset_w(seed, time_limits ? time_limits[b] : (p.mean_time_limit > 0.0 ? sim.sample_time_limit(seed) : INFINITY));
}

// NS: executor slots per lane of the batched fast path (1: E <= 32, 2: E <= 64), see ssb_sim.cuh
template <int NS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, NS == 1 ? SSB_NS1_CTAS : SSB_NS2_CTAS)
k_step(Params p, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask, int max_events,
       int auto_reset, uint64_t seed_step, int32_t *next_a, int32_t *next_n, int dynamic_partition)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    if (mask && !mask[b]) return;
    Sim sim(p, b, lane);
    // next_a / next_n (optional): the built-in fair / FIFO scheduler's action for the observation this call
    // leaves behind (ssb_step_fair_host), evaluated while the state is still in cache
    auto suggest = [&]() {
        if (!next_a) return;
        int a = -1, n = 1;
        if (!sim.h->error && !sim.h->done && !sim.h->pending) sim.fair_action_w(dynamic_partition != 0, a, n);
        if (lane == 0) { next_a[b] = a; next_n[b] = n; }
    };
    if (auto_reset && !sim.h->error && (sim.h->done || sim.oh->truncated)) {
        auto_reset_w(sim, lane, seed_step);
        if (lane == 0) sim.oh->was_reset = 1;
        __syncwarp();
        suggest();
        return;
    }
    if (lane == 0) sim.oh->error = 0;
    __syncwarp();
    sim.template step_w<NS>(stage_idx[b], num_exec[b], max_events);
    __syncwarp();
    suggest();
}

__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
k_fair_actions(Params p, int dynamic_partition, int32_t *stage_idx, int32_t *num_exec)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    Sim sim(p, b, lane);
    int a = -1, n = 1;
    sim.fair_action_w(dynamic_partition != 0, a, n);
    if (lane == 0) { stage_idx[b] = a; num_exec[b] = n; }
}

// fused policy + step: `num_decisions` decisions per environment in one launch
// (min 7 CTAs per SM for the one-slot kernel: 4096 envs = 1024 CTAs must all be resident at once on
// 148 SMs; at 80 registers only 6 fit and the last 136 CTAs run as a second wave, +37 % time.
// Two-slot kernel: 4 CTAs per SM = 128 registers, what it needs without spilling.)
template <int NS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, NS == 1 ? SSB_NS1_CTAS : SSB_NS2_CTAS)
k_rollout_fair(Params p, int num_decisions, int dynamic_partition, int auto_reset, uint64_t seed_step,
               ssb_transition *traj)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    rollout_w<NS>(
        p, b, lane, [](Sim &sim, int dyn, int &a, int &n) { sim.fair_action_w(dyn != 0, a, n); }, dynamic_partition,
        num_decisions, auto_reset, seed_step, traj);
}

// the fixed-duration rollout (ssb_rollout.cuh) with the fair / FIFO policy.  (A kernel of its own, so that the
// default rollout kernel stays as measured.)
template <int NS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, NS == 1 ? SSB_NS1_CTAS : SSB_NS2_CTAS)
k_rollout_fair_async(Params p, int max_decisions, double duration, int dynamic_partition, uint64_t seed_step,
                     ssb_transition *traj, int32_t *num_steps, double *elapsed_out)
{
    const int b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    Sim sim(p, b, lane);
    rollout_async_w<NS>(
        sim, b, lane, [](Sim &sim, int dyn, int &a, int &n) { sim.fair_action_w(dyn != 0, a, n); }, dynamic_partition,
        max_decisions, duration, seed_step, traj, num_steps, elapsed_out);
}

// collect_stats sums in a fixed order: block k reduces the envs k, k + STATS_BLOCKS, ... (one warp per env, lanes
// over its jobs) into part[k][6]; a last warp adds the blocks' partial sums in block order.
constexpr int STATS_BLOCKS = 128;
__global__ void __launch_bounds__(256) k_collect_stats_part(Params p, double *part)
{
    __shared__ double sh[8][6];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double acc[6] = {0, 0, 0, 0, 0, 0};
    for (int b = (int)blockIdx.x + w * STATS_BLOCKS; b < p.B; b += 8 * STATS_BLOCKS) {
        const EnvHdr &h = p.hdr[b];
        const JobRec *jb = p.job + (size_t)b * p.Jc;
        const double wall = h.wall_time;
        double jt = 0.0, cd = 0.0;
        int nc = 0, na = 0;
        for (int j = lane; j < h.next_arrival; j += 32) {  // jobs that have arrived
            const JobRec &J = jb[j];
            jt += fmin(J.t_completed, wall) - J.t_arrival;
            if (J.state == JOB_COMPLETED) { nc++; cd += J.t_completed - J.t_arrival; }
            na++;
        }
        for (int off = 16; off; off >>= 1) {  // fixed butterfly order
            jt += __shfl_xor_sync(0xffffffffu, jt, off);
            cd += __shfl_xor_sync(0xffffffffu, cd, off);
            nc += __shfl_xor_sync(0xffffffffu, nc, off);
            na += __shfl_xor_sync(0xffffffffu, na, off);
        }
        if (wall > 0.0) { acc[0] += jt / wall; acc[1] += 1.0; }
        acc[2] += nc; acc[3] += na; acc[4] += cd; acc[5] += wall;
    }
    if (lane == 0)
        for (int i = 0; i < 6; i++) sh[w][i] = acc[i];
    __syncthreads();
    if (threadIdx.x < 6) {
        double s = 0.0;
        for (int i = 0; i < 8; i++) s += sh[i][threadIdx.x];
        part[(size_t)blockIdx.x * 8 + threadIdx.x] = s;
    }
}
__global__ void k_collect_stats_final(const double *part, double *out)
{
    if (threadIdx.x < 8) {
        double s = 0.0;
        if (threadIdx.x < 6)
            for (int k = 0; k < STATS_BLOCKS; k++) s += part[(size_t)k * 8 + threadIdx.x];
        out[threadIdx.x] = s;
    }
}

// ---- packed observations: the rows of every env's observation back to back (what a host caller copies out)
// offsets[b] = (first node, first edge, first job) of env b in the packed arrays, offsets[B] = the totals.
// One block; every thread scans a contiguous chunk of envs, the chunk sums are scanned through shared memory.
__global__ void __launch_bounds__(1024) k_pack_scan(Params p, int32_t *offsets)
{
    __shared__ int sh[3][1024];
    const int t = threadIdx.x, per = (p.B + 1023) / 1024, lo = min(t * per, p.B), hi = min(lo + per, p.B);
    int sn = 0, se = 0, sj = 0;
    for (int b = lo; b < hi; b++) {
        const ssb_obs_hdr &o = p.obs_hdr[b];
        sn += o.num_nodes; se += o.num_edges; sj += o.num_active_jobs;
    }
    sh[0][t] = sn; sh[1][t] = se; sh[2][t] = sj;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        int a = 0, b2 = 0, c = 0;
        if (t >= off) { a = sh[0][t - off]; b2 = sh[1][t - off]; c = sh[2][t - off]; }
        __syncthreads();
        sh[0][t] += a; sh[1][t] += b2; sh[2][t] += c;
        __syncthreads();
    }
    int on = sh[0][t] - sn, oe = sh[1][t] - se, oj = sh[2][t] - sj;
    for (int b = lo; b < hi; b++) {
        offsets[3 * b] = on; offsets[3 * b + 1] = oe; offsets[3 * b + 2] = oj;
        const ssb_obs_hdr &o = p.obs_hdr[b];
        on += o.num_nodes; oe += o.num_edges; oj += o.num_active_jobs;
    }
    if (t == 1023) { offsets[3 * p.B] = sh[0][t]; offsets[3 * p.B + 1] = sh[1][t]; offsets[3 * p.B + 2] = sh[2][t]; }
}
__global__ void __launch_bounds__(128)
k_pack_copy(Params p, const int32_t *offsets, float *nodes, int32_t *edges, int32_t *dag_ptr, int32_t *supplies)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const ssb_obs_hdr &o = p.obs_hdr[b];
    const int on = offsets[3 * b], oe = offsets[3 * b + 1], oj = offsets[3 * b + 2];
    const float *sn = p.obs_nodes + (size_t)b * p.Sc * 3;
    const int32_t *se = p.obs_edges + (size_t)b * p.Mc * 2;
    for (int i = lane; i < 3 * o.num_nodes; i += 32) nodes[(size_t)on * 3 + i] = sn[i];
    for (int i = lane; i < 2 * o.num_edges; i += 32) edges[(size_t)oe * 2 + i] = se[i];
    for (int i = lane; i <= o.num_active_jobs; i += 32) dag_ptr[oj + b + i] = p.obs_dag_ptr[(size_t)b * (p.Jc + 1) + i];
    for (int i = lane; i < o.num_active_jobs; i += 32) supplies[oj + i] = p.obs_supplies[(size_t)b * p.Jc + i];
}

__global__ void k_zero_stats(ssb_stats *s, int n)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) s[i] = ssb_stats{};
}

// ------------------------------------------------------------------------------------ workspace
int compute_dims(const ssb_config &c, const ssb_bank &bk, Dims &d)
{
    if (c.num_envs < 1 || c.num_executors < 1 || c.num_executors > 128) return SSB_E_INVALID;
    if (c.max_jobs < 1 || c.max_jobs > 16000) return SSB_E_INVALID;
    if (c.job_arrival_cap > c.max_jobs) return SSB_E_INVALID;
    if (!(c.job_arrival_rate > 0)) return SSB_E_INVALID;
    if (bk.num_templates != 154) return SSB_E_INVALID;  // 7 sizes x 22 queries (tpch.py:14-15)
    int ms = 0, me = 0;
    for (int t = 0; t < bk.num_templates; t++) {
        ms = bk.num_stages[t] > ms ? bk.num_stages[t] : ms;
        int ne = bk.edge_base[t + 1] - bk.edge_base[t];
        me = ne > me ? ne : me;
    }
    if (ms < 1 || ms > 64) return SSB_E_INVALID;
    d.max_stages = ms;
    d.max_edges = me;
    d.TAB = 8;
    while (d.TAB <= 4 * c.num_executors) d.TAB <<= 1;
    d.RT = 8;
    while (d.RT <= 4 * c.max_jobs) d.RT <<= 1;
    d.Sc = c.max_jobs * ms;
    d.Mc = c.max_jobs * me;
    if (d.Sc > 32000) return SSB_E_INVALID;
    d.P = 2 + c.max_jobs + d.Sc;
    d.Cc = 2 * c.num_executors + 16;
    return SSB_OK;
}

void carve(Carver &cv, const ssb_config &c, const ssb_bank &bk, const Dims &d, Params &p, BankDev &bd,
           int32_t **st_a, int32_t **st_n, uint64_t **st_seed, double **st_tl, uint8_t **st_mask, uint32_t **pol_streams)
{
    const size_t B = c.num_envs, T = bk.num_templates, TS = bk.num_template_stages;
    bd.num_stages = cv.take<int32_t>(T);
    bd.stage_base = cv.take<int32_t>(T + 1);
    bd.edge_base = cv.take<int32_t>(T + 1);
    bd.num_tasks = cv.take<int32_t>(TS);
    bd.edges = cv.take<int16_t>(2 * (size_t)bk.num_template_edges);
    bd.rough = cv.take<double>(TS);
    bd.parent = cv.take<uint64_t>(TS);
    bd.child = cv.take<uint64_t>(TS);
    bd.present = cv.take<uint8_t>(TS * 4);
    bd.dur = cv.take<uint2>(TS * 24);
    bd.vals = cv.take<double>((size_t)bk.num_values + 1);
    bd.iv = cv.take<short4>((size_t)c.num_executors + 1);
    p.hdr = cv.take<EnvHdr>(B);
    p.exec = cv.take<ExecRec>(B * c.num_executors);
    p.job = cv.take<JobRec>(B * c.max_jobs);
    p.stage = cv.take<StageRec>(B * d.Sc);
    p.active = cv.take<int16_t>(B * c.max_jobs);
    p.old_act = cv.take<int16_t>(B * c.max_jobs);
    p.reward_ord = cv.take<int16_t>(B * c.max_jobs);
    p.commits = cv.take<Commit>(B * d.Cc);
    p.pool_hdr = cv.take<PoolHdr>(B * d.P);
    p.pool_tab = cv.take<uint8_t>(B * d.P * d.TAB);
    p.scr_tab = cv.take<uint8_t>(B * 3 * d.TAB);
    p.rset = cv.take<uint16_t>(B * 2 * d.RT);
    p.trace_t = cv.take<double>(c.tape_capacity > 0 ? B * c.max_jobs : 1);
    p.trace_tmpl = cv.take<int32_t>(c.tape_capacity > 0 ? B * c.max_jobs : 1);
    p.tape = cv.take<double>(c.tape_capacity > 0 ? B * (size_t)c.tape_capacity : 1);
    p.log = cv.take<LogRow>(c.log_capacity > 0 ? B * (size_t)c.log_capacity : 1);
    p.hist = cv.take<HistRow>(c.history_capacity > 0 ? B * (size_t)c.history_capacity : 1);
    p.stats = cv.take<ssb_stats>(B);
    p.stats_part = cv.take<double>(128 * 8);
    p.prof = cv.take<unsigned long long>(B * 16);
    p.obs_hdr = cv.take<ssb_obs_hdr>(B);
    p.obs_nodes = cv.take<float>(B * d.Sc * 3);
    p.obs_edges = cv.take<int32_t>(B * d.Mc * 2);
    p.obs_dag_ptr = cv.take<int32_t>(B * (c.max_jobs + 1));
    p.obs_supplies = cv.take<int32_t>(B * c.max_jobs);
    if (c.flags & (SSB_FLAG_DECIMA_OBS | SSB_FLAG_DECIMA_POLICY)) {
        p.dec_feat = cv.take<float>(B * d.Sc * 5);
        p.dec_stage_mask = cv.take<uint8_t>(B * d.Sc);
        p.dec_frontier_mask = cv.take<uint8_t>(B * d.Sc);
        p.dec_caps = cv.take<int32_t>(B * c.max_jobs);
        p.dec_edge_bits = cv.take<uint64_t>(B * d.Mc);
        p.dec_depth = cv.take<int32_t>(B);
    }
    if (c.flags & SSB_FLAG_DECIMA_POLICY) ssb_i_policy_carve(cv, c, d, p, pol_streams);
    *st_a = cv.take<int32_t>(B);
    *st_n = cv.take<int32_t>(B);
    *st_seed = cv.take<uint64_t>(B);
    *st_tl = cv.take<double>(B);
    *st_mask = cv.take<uint8_t>(B);
}

}  // namespace

static int host_begin(ssb_env *env)
{
    CUDA_TRY(cudaSetDevice(env->device));
    if (env->dirty) {
        CUDA_TRY(cudaStreamWaitEvent(env->own_stream, env->ev_last, 0));
        env->dirty = 0;
    }
    return SSB_OK;
}

extern "C" {

int ssb_abi_version(void) { return SSB_ABI_VERSION; }
const char *ssb_last_cuda_error(void) { return g_cuda_err; }

int ssb_workspace_bytes(const ssb_config *cfg, const ssb_bank *bank, size_t *bytes)
{
    if (!cfg || !bank || !bytes) return SSB_E_INVALID;
    Dims d;
    int rc = compute_dims(*cfg, *bank, d);
    if (rc) return rc;
    Carver cv{nullptr};
    Params p{};
    BankDev bd{};
    int32_t *a, *n; uint64_t *s; double *tl; uint8_t *m; uint32_t *ps;
    carve(cv, *cfg, *bank, d, p, bd, &a, &n, &s, &tl, &m, &ps);
    *bytes = (cv.off + 255) & ~size_t(255);
    return SSB_OK;
}

int ssb_create(const ssb_config *cfg, const ssb_bank *bk, int device, void *workspace,
               size_t workspace_bytes, ssb_env **out)
{
    if (!cfg || !bk || !workspace || !out) return SSB_E_INVALID;
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return SSB_E_WORKSPACE;
    Dims d;
    int rc = compute_dims(*cfg, *bk, d);
    if (rc) return rc;
    size_t need = 0;
    ssb_workspace_bytes(cfg, bk, &need);
    if (workspace_bytes < need) return SSB_E_WORKSPACE;
    CUDA_TRY(cudaSetDevice(device));
    ssb_env *env = new (std::nothrow) ssb_env();
    if (!env) return SSB_E_INVALID;
    env->cfg = *cfg;
    env->dims = d;
    env->device = device;
    env->ws = static_cast<char *>(workspace);
    env->ws_bytes = workspace_bytes;
    Carver cv{env->ws};
    Params &p = env->p;
    p = Params{};
    carve(cv, *cfg, *bk, d, p, env->bank, &env->st_a, &env->st_n, &env->st_seed, &env->st_tl, &env->st_mask,
          &env->pol_streams);
    p.B = cfg->num_envs; p.E = cfg->num_executors; p.Jc = cfg->max_jobs; p.Sc = d.Sc; p.Mc = d.Mc;
    p.TAB = d.TAB; p.RT = d.RT; p.P = d.P; p.Cc = d.Cc; p.max_stages = d.max_stages;
    p.tape_cap = cfg->tape_capacity; p.log_cap = cfg->log_capacity;
    p.hist_cap = cfg->history_capacity > 0 ? cfg->history_capacity : 0;
    p.job_arrival_cap = cfg->job_arrival_cap;
    p.moving_delay = cfg->moving_delay; p.warmup_delay = cfg->warmup_delay;
    p.mean_interarrival = 1 / cfg->job_arrival_rate;  // tpch.py:42
    p.beta = cfg->beta;
    env->grid = (cfg->num_envs + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    {
        const char *ng = getenv("SSB_NO_GRAPH");
        env->no_graph = ng && ng[0] == '1';
    }
    CUDA_TRY(cudaDeviceGetAttribute(&env->num_sms, cudaDevAttrMultiProcessorCount, device));
    {
        // longest chain of topological generations over the templates bounds the depth of every observation
        int dmax = 0;
        for (int t = 0; t < bk->num_templates; t++) {
            const int ns = bk->num_stages[t], base = bk->stage_base[t];
            const uint64_t all = ns >= 64 ? ~0ull : ((1ull << ns) - 1);
            uint64_t done = 0;
            int gens = 0;
            while (done != all && gens < 64) {
                uint64_t lk = 0;
                for (int s = 0; s < ns; s++)
                    if (!((done >> s) & 1) && (bk->parent_mask[base + s] & ~done) == 0) lk |= 1ull << s;
                if (!lk) break;
                done |= lk;
                gens++;
            }
            dmax = gens - 1 > dmax ? gens - 1 : dmax;
        }
        env->dmax = dmax;
    }
    if (p.pol_w) {
        const int rc = ssb_i_policy_init(env);
        if (rc) return rc;
    }
    // ---- bank upload
    const size_t T = bk->num_templates, TS = bk->num_template_stages, ME = bk->num_template_edges;
    BankDev &bd = env->bank;
    CUDA_TRY(cudaMemcpy(bd.num_stages, bk->num_stages, T * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.stage_base, bk->stage_base, (T + 1) * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.edge_base, bk->edge_base, (T + 1) * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.num_tasks, bk->num_tasks, TS * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.rough, bk->rough_duration, TS * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.parent, bk->parent_mask, TS * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.child, bk->child_mask, TS * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(bd.vals, bk->dur_values, (size_t)bk->num_values * 8, cudaMemcpyHostToDevice));
    {
        std::vector<int16_t> e16(2 * ME);
        for (size_t i = 0; i < 2 * ME; i++) e16[i] = (int16_t)bk->edges[i];
        CUDA_TRY(cudaMemcpy(bd.edges, e16.data(), e16.size() * 2, cudaMemcpyHostToDevice));
        std::vector<uint8_t> pr(TS * 4, 0);
        for (size_t i = 0; i < TS; i++)
            for (int w = 0; w < 3; w++) pr[i * 4 + w] = bk->present[i * 3 + w];
        CUDA_TRY(cudaMemcpy(bd.present, pr.data(), pr.size(), cudaMemcpyHostToDevice));
        std::vector<uint2> du(TS * 24);
        for (size_t i = 0; i < TS * 24; i++) du[i] = make_uint2(bk->dur_off[i], bk->dur_cnt[i]);
        CUDA_TRY(cudaMemcpy(bd.dur, du.data(), du.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        for (size_t i = 0; i < TS; i++)
            if (bk->num_tasks[i] < 1 || bk->num_tasks[i] > 65535) { delete env; return SSB_E_INVALID; }
        // _init_executor_intervals (tpch.py:237-262) as integer levels
        const int LV[8] = {5, 10, 20, 40, 50, 60, 80, 100};
        const int cap = cfg->num_executors;
        std::vector<int16_t> iv(2 * (cap + 1), 0);
        for (int i = 0; i <= LV[0] && i <= cap; i++) iv[2 * i] = iv[2 * i + 1] = LV[0];
        for (int i = 0; i < 7; i++) {
            for (int r = LV[i] + 1; r < LV[i + 1] && r <= cap; r++) { iv[2 * r] = LV[i]; iv[2 * r + 1] = LV[i + 1]; }
            if (LV[i + 1] > cap) break;
            iv[2 * LV[i + 1]] = iv[2 * LV[i + 1] + 1] = LV[i + 1];
        }
        if (cap > LV[7]) for (int r = LV[7] + 1; r < cap; r++) iv[2 * r] = iv[2 * r + 1] = LV[7];
        std::vector<short4> iv4(cap + 1);
        for (int r = 0; r <= cap; r++) {
            int li = -1, ri = -1;  // level value -> level index (-1: not a data level, e.g. the 0 rows)
            for (int q = 0; q < 8; q++) {
                if (LV[q] == iv[2 * r]) li = q;
                if (LV[q] == iv[2 * r + 1]) ri = q;
            }
            iv4[r] = make_short4(iv[2 * r], iv[2 * r + 1], (short)li, (short)ri);
        }
        CUDA_TRY(cudaMemcpy(bd.iv, iv4.data(), iv4.size() * sizeof(short4), cudaMemcpyHostToDevice));
    }
    p.b_num_stages = bd.num_stages; p.b_stage_base = bd.stage_base; p.b_edge_base = bd.edge_base;
    p.b_num_tasks = bd.num_tasks; p.b_edges = bd.edges; p.b_rough = bd.rough; p.b_parent = bd.parent;
    p.b_child = bd.child; p.b_present = bd.present; p.b_dur = bd.dur; p.b_vals = bd.vals; p.iv = bd.iv;
    CUDA_TRY(cudaMemset(p.hdr, 0, sizeof(EnvHdr) * (size_t)p.B));
    CUDA_TRY(cudaMemset(p.stats, 0, sizeof(ssb_stats) * (size_t)p.B));
    CUDA_TRY(cudaMemset(p.prof, 0, sizeof(unsigned long long) * 16 * (size_t)p.B));
    CUDA_TRY(cudaMemset(p.obs_hdr, 0, sizeof(ssb_obs_hdr) * (size_t)p.B));
    CUDA_TRY(cudaStreamCreateWithFlags(&env->own_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&env->ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&env->ev_last, cudaEventDisableTiming));
    CUDA_TRY(cudaDeviceSynchronize());
    *out = env;
    return SSB_OK;
}

int ssb_destroy(ssb_env *env)
{
    if (!env) return SSB_E_INVALID;
    cudaSetDevice(env->device);
    cudaStreamSynchronize(env->own_stream);
    cudaStreamDestroy(env->own_stream);
    if (env->dg_exec) cudaGraphExecDestroy(env->dg_exec);
    if (env->ev) cudaEventDestroy(env->ev);
    if (env->ev_last) cudaEventDestroy(env->ev_last);
    delete env;
    return SSB_OK;
}

int ssb_load_trace(ssb_env *env, int32_t b, int32_t n_jobs, const double *t_arrival, const int32_t *tmpl,
                   const double *tape, int64_t n_tape)
{
    if (!env || b < 0 || b >= env->p.B || n_jobs < 1 || n_jobs > env->p.Jc || !t_arrival || !tmpl)
        return SSB_E_INVALID;
    if (env->cfg.tape_capacity <= 0) return SSB_E_INVALID;
    if (tape && n_tape > env->cfg.tape_capacity) return SSB_E_INVALID;
    if (t_arrival[0] != 0.0) return SSB_E_INVALID;  // spark_sched_sim.py:150
    for (int j = 0; j < n_jobs; j++)
        if (tmpl[j] < 0 || tmpl[j] >= 154) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    const Params &p = env->p;
    CUDA_TRY(cudaMemcpy(p.trace_t + (size_t)b * p.Jc, t_arrival, n_jobs * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(p.trace_tmpl + (size_t)b * p.Jc, tmpl, n_jobs * 4, cudaMemcpyHostToDevice));
    int32_t tl = tape ? (int32_t)n_tape : -1;
    if (tape && n_tape > 0)
        CUDA_TRY(cudaMemcpy(p.tape + (size_t)b * p.tape_cap, tape, n_tape * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(&p.hdr[b].trace_jobs, &n_jobs, 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(&p.hdr[b].tape_len, &tl, 4, cudaMemcpyHostToDevice));
    return SSB_OK;
}

int ssb_clear_trace(ssb_env *env, int32_t b)
{
    if (!env || b < 0 || b >= env->p.B) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    int32_t z = 0;
    CUDA_TRY(cudaMemcpy(&env->p.hdr[b].trace_jobs, &z, 4, cudaMemcpyHostToDevice));
    return SSB_OK;
}

int ssb_reset(ssb_env *env, const uint64_t *seeds, const double *time_limits, const uint8_t *mask, void *stream)
{
    if (!env) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    k_reset<<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(env->p, seeds, time_limits, mask);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_i_step_launch(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
                      int32_t max_events, int32_t *next_a, int32_t *next_n, int dyn, cudaStream_t s,
                      int force_autoreset, uint64_t force_seed_step)
{
    const int ar = force_autoreset ? 1 : env->auto_reset;
    const uint64_t ss = force_autoreset ? force_seed_step : env->auto_seed_step;
    if (env->p.E <= 32)
        k_step<1><<<env->grid, WARPS_PER_CTA * 32, 0, s>>>(env->p, stage_idx, num_exec, mask, max_events, ar, ss, next_a,
                                                           next_n, dyn);
    else
        k_step<2><<<env->grid, WARPS_PER_CTA * 32, 0, s>>>(env->p, stage_idx, num_exec, mask, max_events, ar, ss, next_a,
                                                           next_n, dyn);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, s);
    return SSB_OK;
}

int ssb_step(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
             int32_t max_events, void *stream)
{
    if (!env || !stage_idx || !num_exec) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    return ssb_i_step_launch(env, stage_idx, num_exec, mask, max_events, nullptr, nullptr, 0, (cudaStream_t)stream, 0, 0);
}

int ssb_set_autoreset(ssb_env *env, int32_t enable, uint64_t seed_step)
{
    if (!env) return SSB_E_INVALID;
    env->auto_reset = enable ? 1 : 0;
    env->auto_seed_step = seed_step;
    ssb_i_drop_decision_graph(env);
    return SSB_OK;
}

int ssb_set_mean_time_limit(ssb_env *env, double mean_ms)
{
    if (!env || !(mean_ms >= 0.0)) return SSB_E_INVALID;
    env->p.mean_time_limit = mean_ms;
    ssb_i_drop_decision_graph(env);
    return SSB_OK;
}

int ssb_reset_host(ssb_env *env, const uint64_t *seeds, const double *time_limits, const uint8_t *mask,
                   ssb_obs_hdr *hdr_out)
{
    if (!env) return SSB_E_INVALID;
    {
        const int rcb = host_begin(env);  // also waits for work still queued on the caller's streams
        if (rcb) return rcb;
    }
    cudaStream_t s = env->own_stream;
    const size_t B = env->p.B;
    if (seeds) CUDA_TRY(cudaMemcpyAsync(env->st_seed, seeds, B * 8, cudaMemcpyHostToDevice, s));
    if (time_limits) CUDA_TRY(cudaMemcpyAsync(env->st_tl, time_limits, B * 8, cudaMemcpyHostToDevice, s));
    if (mask) CUDA_TRY(cudaMemcpyAsync(env->st_mask, mask, B, cudaMemcpyHostToDevice, s));
    int rc = ssb_reset(env, seeds ? env->st_seed : nullptr, time_limits ? env->st_tl : nullptr,
                       mask ? env->st_mask : nullptr, s);
    if (rc) return rc;
    if (hdr_out) CUDA_TRY(cudaMemcpyAsync(hdr_out, env->p.obs_hdr, B * sizeof(ssb_obs_hdr), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return SSB_OK;
}

int ssb_step_host(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
                  int32_t max_events, ssb_obs_hdr *hdr_out)
{
    if (!env || !stage_idx || !num_exec) return SSB_E_INVALID;
    {
        const int rcb = host_begin(env);  // also waits for work still queued on the caller's streams
        if (rcb) return rcb;
    }
    cudaStream_t s = env->own_stream;
    const size_t B = env->p.B;
    CUDA_TRY(cudaMemcpyAsync(env->st_a, stage_idx, B * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(env->st_n, num_exec, B * 4, cudaMemcpyHostToDevice, s));
    if (mask) CUDA_TRY(cudaMemcpyAsync(env->st_mask, mask, B, cudaMemcpyHostToDevice, s));
    int rc = ssb_step(env, env->st_a, env->st_n, mask ? env->st_mask : nullptr, max_events, s);
    if (rc) return rc;
    if (hdr_out) CUDA_TRY(cudaMemcpyAsync(hdr_out, env->p.obs_hdr, B * sizeof(ssb_obs_hdr), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return SSB_OK;
}

int ssb_step_fair_host(ssb_env *env, const int32_t *stage_idx, const int32_t *num_exec, const uint8_t *mask,
                       int32_t max_events, int32_t dynamic_partition, ssb_obs_hdr *hdr_out, int32_t *next_stage_idx,
                       int32_t *next_num_exec)
{
    if (!env || !stage_idx || !num_exec || !next_stage_idx || !next_num_exec) return SSB_E_INVALID;
    {
        const int rcb = host_begin(env);  // also waits for work still queued on the caller's streams
        if (rcb) return rcb;
    }
    cudaStream_t s = env->own_stream;
    const size_t B = env->p.B;
    CUDA_TRY(cudaMemcpyAsync(env->st_a, stage_idx, B * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(env->st_n, num_exec, B * 4, cudaMemcpyHostToDevice, s));
    if (mask) CUDA_TRY(cudaMemcpyAsync(env->st_mask, mask, B, cudaMemcpyHostToDevice, s));
    // the suggestions are written to the staging arrays the actions were read from (each env reads its action
    // before it writes its suggestion)
    int rc = ssb_i_step_launch(env, env->st_a, env->st_n, mask ? env->st_mask : nullptr, max_events, env->st_a, env->st_n,
                               dynamic_partition, s, 0, 0);
    if (rc) return rc;
    if (hdr_out) CUDA_TRY(cudaMemcpyAsync(hdr_out, env->p.obs_hdr, B * sizeof(ssb_obs_hdr), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(next_stage_idx, env->st_a, B * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(next_num_exec, env->st_n, B * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return SSB_OK;
}

// layout of the caller's scratch for the packed observation
namespace {
struct PackLayout { size_t off_offsets, off_nodes, off_edges, off_dag, off_sup, bytes; };
PackLayout pack_layout(const Params &p)
{
    PackLayout l{};
    size_t o = 0;
    auto take = [&](size_t n) { size_t at = o; o += (n + 255) & ~size_t(255); return at; };
    l.off_offsets = take(sizeof(int32_t) * 3 * ((size_t)p.B + 1));
    l.off_nodes = take(sizeof(float) * 3 * (size_t)p.B * p.Sc);
    l.off_edges = take(sizeof(int32_t) * 2 * (size_t)p.B * p.Mc);
    l.off_dag = take(sizeof(int32_t) * (size_t)p.B * (p.Jc + 1));
    l.off_sup = take(sizeof(int32_t) * (size_t)p.B * p.Jc);
    l.bytes = o;
    return l;
}
}  // namespace

int ssb_packed_obs_bytes(ssb_env *env, size_t *bytes)
{
    if (!env || !bytes) return SSB_E_INVALID;
    *bytes = pack_layout(env->p).bytes;
    return SSB_OK;
}

int ssb_get_obs_host(ssb_env *env, ssb_packed_obs *out, void *scratch, size_t scratch_bytes)
{
    if (!env || !out || !out->offsets || !scratch || (reinterpret_cast<uintptr_t>(scratch) & 255)) return SSB_E_INVALID;
    const Params &p = env->p;
    const PackLayout l = pack_layout(p);
    if (scratch_bytes < l.bytes) return SSB_E_WORKSPACE;
    {
        const int rcb = host_begin(env);  // also waits for work still queued on the caller's streams
        if (rcb) return rcb;
    }
    cudaStream_t s = env->own_stream;
    char *sc = static_cast<char *>(scratch);
    int32_t *d_off = reinterpret_cast<int32_t *>(sc + l.off_offsets);
    float *d_nodes = reinterpret_cast<float *>(sc + l.off_nodes);
    int32_t *d_edges = reinterpret_cast<int32_t *>(sc + l.off_edges), *d_dag = reinterpret_cast<int32_t *>(sc + l.off_dag),
            *d_sup = reinterpret_cast<int32_t *>(sc + l.off_sup);
    k_pack_scan<<<1, 1024, 0, s>>>(p, d_off);
    k_pack_copy<<<(p.B + 3) / 4, 128, 0, s>>>(p, d_off, d_nodes, d_edges, d_dag, d_sup);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out->offsets, d_off, sizeof(int32_t) * 3 * ((size_t)p.B + 1), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));  // the totals size the copies below
    const int64_t tn = out->offsets[3 * p.B], te = out->offsets[3 * p.B + 1], tj = out->offsets[3 * p.B + 2];
    if (tn > out->node_capacity || te > out->edge_capacity || tj > out->job_capacity) return SSB_E_WORKSPACE;
    if (out->nodes) CUDA_TRY(cudaMemcpyAsync(out->nodes, d_nodes, sizeof(float) * 3 * tn, cudaMemcpyDeviceToHost, s));
    if (out->edge_links) CUDA_TRY(cudaMemcpyAsync(out->edge_links, d_edges, sizeof(int32_t) * 2 * te, cudaMemcpyDeviceToHost, s));
    if (out->dag_ptr) CUDA_TRY(cudaMemcpyAsync(out->dag_ptr, d_dag, sizeof(int32_t) * (tj + p.B), cudaMemcpyDeviceToHost, s));
    if (out->exec_supplies) CUDA_TRY(cudaMemcpyAsync(out->exec_supplies, d_sup, sizeof(int32_t) * tj, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return SSB_OK;
}

int ssb_rollout_fair_traj(ssb_env *env, int32_t num_decisions, int32_t dynamic_partition, int32_t auto_reset,
                          uint64_t seed_step, ssb_transition *traj, void *stream)
{
    if (!env || num_decisions < 0) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    if (env->p.E <= 32)
        k_rollout_fair<1><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(
            env->p, num_decisions, dynamic_partition, auto_reset, seed_step, traj);
    else
        k_rollout_fair<2><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(
            env->p, num_decisions, dynamic_partition, auto_reset, seed_step, traj);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_rollout_fair_async(ssb_env *env, int32_t max_decisions, double rollout_duration, int32_t dynamic_partition,
                           uint64_t seed_step, ssb_transition *traj, int32_t *num_steps, double *elapsed, void *stream)
{
    if (!env || max_decisions < 0 || !(rollout_duration > 0.0)) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    if (env->p.E <= 32)
        k_rollout_fair_async<1><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(
            env->p, max_decisions, rollout_duration, dynamic_partition, seed_step, traj, num_steps, elapsed);
    else
        k_rollout_fair_async<2><<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(
            env->p, max_decisions, rollout_duration, dynamic_partition, seed_step, traj, num_steps, elapsed);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_rollout_fair(ssb_env *env, int32_t num_decisions, int32_t dynamic_partition, int32_t auto_reset,
                     uint64_t seed_step, void *stream)
{
    return ssb_rollout_fair_traj(env, num_decisions, dynamic_partition, auto_reset, seed_step, nullptr, stream);
}

int ssb_fair_actions(ssb_env *env, int32_t dynamic_partition, int32_t *stage_idx, int32_t *num_exec, void *stream)
{
    if (!env || !stage_idx || !num_exec) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    k_fair_actions<<<env->grid, WARPS_PER_CTA * 32, 0, (cudaStream_t)stream>>>(env->p, dynamic_partition,
                                                                               stage_idx, num_exec);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_get_views(ssb_env *env, ssb_views *out)
{
    if (!env || !out) return SSB_E_INVALID;
    out->hdr = env->p.obs_hdr;
    out->nodes = env->p.obs_nodes;
    out->edge_links = env->p.obs_edges;
    out->dag_ptr = env->p.obs_dag_ptr;
    out->exec_supplies = env->p.obs_supplies;
    out->node_stride = env->p.Sc;
    out->edge_stride = env->p.Mc;
    out->job_stride = env->p.Jc;
    out->pad = 0;
    return SSB_OK;
}

int ssb_decima_obs(ssb_env *env, void *stream)
{
    if (!env || !env->p.dec_feat) return SSB_E_INVALID;  // needs SSB_FLAG_DECIMA_OBS
    SSB_ON_DEVICE(env);
    const int rc = ssb_i_decima_obs(env, (cudaStream_t)stream);
    if (rc) return rc;
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_get_decima_views(ssb_env *env, ssb_decima_views *out)
{
    if (!env || !out || !env->p.dec_feat) return SSB_E_INVALID;
    out->features = env->p.dec_feat;
    out->stage_mask = env->p.dec_stage_mask;
    out->frontier_mask = env->p.dec_frontier_mask;
    out->commit_caps = env->p.dec_caps;
    out->edge_bits = env->p.dec_edge_bits;
    out->depth = env->p.dec_depth;
    out->node_stride = env->p.Sc;
    out->edge_stride = env->p.Mc;
    out->job_stride = env->p.Jc;
    out->pad = 0;
    return SSB_OK;
}

int ssb_get_stats(ssb_env *env, ssb_stats **out)
{
    if (!env || !out) return SSB_E_INVALID;
    *out = env->p.stats;
    return SSB_OK;
}

int ssb_get_debug_counters(ssb_env *env, uint64_t **out)
{
    if (!env || !out) return SSB_E_INVALID;
    *out = reinterpret_cast<uint64_t *>(env->p.prof);
    return SSB_OK;
}

int ssb_collect_stats(ssb_env *env, double *out, void *stream)
{
    if (!env || !out) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    k_collect_stats_part<<<STATS_BLOCKS, 256, 0, (cudaStream_t)stream>>>(env->p, env->p.stats_part);
    k_collect_stats_final<<<1, 32, 0, (cudaStream_t)stream>>>(env->p.stats_part, out);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_reset_stats(ssb_env *env, void *stream)
{
    if (!env) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    k_zero_stats<<<(env->p.B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(env->p.stats, env->p.B);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_get_jobs(ssb_env *env, int32_t b, int32_t *n_jobs, double *t_arrival, double *t_completed,
                 int32_t *tmpl, uint8_t *state, int32_t capacity)
{
    if (!env || b < 0 || b >= env->p.B || !n_jobs) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    CUDA_TRY(cudaDeviceSynchronize());
    EnvHdr h;
    CUDA_TRY(cudaMemcpy(&h, env->p.hdr + b, sizeof(EnvHdr), cudaMemcpyDeviceToHost));
    *n_jobs = h.n_jobs;
    int n = h.n_jobs < capacity ? h.n_jobs : capacity;
    std::vector<JobRec> jr(n > 0 ? n : 1);
    if (n > 0)
        CUDA_TRY(cudaMemcpy(jr.data(), env->p.job + (size_t)b * env->p.Jc, sizeof(JobRec) * n, cudaMemcpyDeviceToHost));
    for (int j = 0; j < n; j++) {
        if (t_arrival) t_arrival[j] = jr[j].t_arrival;
        if (t_completed) t_completed[j] = jr[j].t_completed;
        if (tmpl) tmpl[j] = jr[j].tmpl;
        if (state) state[j] = jr[j].state;
    }
    return SSB_OK;
}

int ssb_get_history(ssb_env *env, int32_t b, int64_t *n_rows, double *t, int16_t *exec, int16_t *job, int64_t capacity)
{
    if (!env || b < 0 || b >= env->p.B || !n_rows) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    CUDA_TRY(cudaDeviceSynchronize());
    EnvHdr h;
    CUDA_TRY(cudaMemcpy(&h, env->p.hdr + b, sizeof(EnvHdr), cudaMemcpyDeviceToHost));
    *n_rows = h.hist_n;
    int64_t n = std::min<int64_t>(std::min<int64_t>(h.hist_n, env->p.hist_cap), capacity);
    if (n <= 0) return SSB_OK;
    std::vector<HistRow> rows(n);
    CUDA_TRY(cudaMemcpy(rows.data(), env->p.hist + (size_t)b * env->p.hist_cap, sizeof(HistRow) * n,
                        cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n; i++) {
        if (t) t[i] = rows[i].t;
        if (exec) exec[i] = rows[i].exec;
        if (job) job[i] = rows[i].job;
    }
    return SSB_OK;
}

int ssb_get_log(ssb_env *env, int32_t b, int64_t lo, int64_t hi, int64_t *n_rows, double *t, uint8_t *type,
                int16_t *job, int16_t *stage, int32_t *task, int16_t *exec, double *t_accepted)
{
    if (!env || b < 0 || b >= env->p.B || !n_rows) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    CUDA_TRY(cudaDeviceSynchronize());
    EnvHdr h;
    CUDA_TRY(cudaMemcpy(&h, env->p.hdr + b, sizeof(EnvHdr), cudaMemcpyDeviceToHost));
    *n_rows = h.log_n;
    if (hi <= lo) return SSB_OK;
    if (env->p.log_cap <= 0 || lo < 0 || hi > h.log_n || hi > env->p.log_cap) return SSB_E_INVALID;
    std::vector<LogRow> rows(hi - lo);
    CUDA_TRY(cudaMemcpy(rows.data(), env->p.log + (size_t)b * env->p.log_cap + lo, sizeof(LogRow) * (hi - lo),
                        cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < hi - lo; i++) {
        const LogRow &r = rows[i];
        if (t) t[i] = r.t;
        if (type) type[i] = r.type;
        if (job) job[i] = r.job;
        if (stage) stage[i] = r.stage;
        if (task) task[i] = r.task;
        if (exec) exec[i] = r.exec;
        if (t_accepted) t_accepted[i] = r.t_acc;
    }
    return SSB_OK;
}

}  // extern "C"

