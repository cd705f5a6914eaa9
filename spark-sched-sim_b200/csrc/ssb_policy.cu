// ssb_policy.cu -- the Decima policy's side of the C ABI (include/ssb.h): weights, the policy call (row lists + tile
// kernels, or the fused kernel), stored observations and their re-evaluation, the backward pass, Decima rollouts.
// A translation unit of its own so that nothing here sits next to the simulator kernels (see ssb_env.cuh).
#define SSB_DECIMA_CTA_ADAPTER
#include "ssb_env.cuh"
#include "ssb_decima.cuh"
#include "ssb_decima_tc.cuh"
#include "ssb_decima_fused.cuh"
#include "ssb_backward.cuh"

using namespace ssb;

namespace {
// The observation adapter (DecimaObsWrapper.observation + make_dag_layer_edge_masks), one CTA per environment:
// pass 1, one thread per active job: the job's edge count in the observation; an exclusive scan gives every job's
// first edge entry (its first node row is the observation's dag_ptr); pass 2: the CTA's warps take the jobs
// round-robin (Sim::decima_obs_job_w).  Same outputs as Sim::decima_obs_w (one warp per env, jobs one after the
// other), which the fused policy kernel runs.
constexpr int ADAPTER_WARPS = 4;
__global__ void __launch_bounds__(ADAPTER_WARPS * 32) k_decima_obs_cta(Params p)
{
    extern __shared__ __align__(16) unsigned char ad_smem[];  // AdJob [Jc], then edge_off int32 [Jc]
    __shared__ uint64_t Sk[ADAPTER_WARPS][64];
    __shared__ int depth_s, scan_s[ADAPTER_WARPS];
    const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    Sim sim(p, b, lane);
    Sim::AdJob *aj = reinterpret_cast<Sim::AdJob *>(ad_smem);
    int32_t *edge_off = reinterpret_cast<int32_t *>(aj + p.Jc);
    const int n_active = sim.h->n_active;
    if (tid == 0) depth_s = 0;
    // pass 1 + block-wide exclusive scan of the edge counts, 128 jobs at a time
    int carry = 0;
    for (int i0 = 0; i0 < n_active; i0 += ADAPTER_WARPS * 32) {
        const int i = i0 + tid;
        int c = 0;
        if (i < n_active) { aj[i] = sim.decima_job_fetch(i); c = aj[i].n_edges; }
        int incl = c;
        for (int off = 1; off < 32; off <<= 1) { const int v = __shfl_up_sync(FULL, incl, off); if (lane >= off) incl += v; }
        if (lane == 31) scan_s[warp] = incl;
        __syncthreads();
        int base = carry;
        for (int w = 0; w < warp; w++) base += scan_s[w];
        if (i < n_active) edge_off[i] = base + incl - c;
        for (int w = 0; w < ADAPTER_WARPS; w++) carry += scan_s[w];
        __syncthreads();
    }
    const int ncommit = sim.num_committable(), src_job = sim.source_job_id();
    const int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
    int D = 0;
    for (int i = warp; i < n_active; i += ADAPTER_WARPS)
        D = max(D, sim.decima_obs_job_w(aj[i], i, dag_ptr[i], edge_off[i], ncommit, src_job, Sk[warp]));
    if (lane == 0 && D) atomicMax(&depth_s, D);
    __syncthreads();
    if (tid == 0) p.dec_depth[b] = depth_s > 1 ? depth_s - 1 : 0;
}

// rollout-buffer rows around one { policy ; step } call of ssb_rollout_decima
// (the row index d lives in device memory so that one captured graph serves every decision of a call)
__global__ void k_traj_pre(Params p, const int32_t *a, const int32_t *n, ssb_transition *traj, int K)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B) return;
    const int d = *p.traj_d;
    ssb_transition t;
    t.wall_time = p.obs_hdr[b].wall_time; t.reward = 0.0; t.stage_idx = a[b]; t.num_exec = n[b];
    t.flags = p.obs_hdr[b].was_reset ? 4 : 0;
    t.lgprob = p.pol_lgprob[b];
    traj[(size_t)b * K + d] = t;
}
__global__ void k_traj_post(Params p, ssb_transition *traj, int K)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B) return;
    const int d = *p.traj_d;
    const ssb_obs_hdr &o = p.obs_hdr[b];
    ssb_transition &t = traj[(size_t)b * K + d];
    if (o.was_reset || o.error == SSB_ENV_DONE) { t.flags = 8; t.reward = 0.0; return; }
    t.reward = o.reward;
    t.flags |= (o.terminated ? 1 : 0) | (o.truncated ? 2 : 0);
}

}  // namespace

void ssb_i_policy_carve(Carver &cv, const ssb_config &c, const Dims &d, Params &p, uint32_t **pol_streams)
{
    const size_t B = c.num_envs;
    {
        p.Epad = (c.num_executors + 3) & ~3;
        p.pol_w = cv.take<float>(dd::TOTAL);
        p.pol_h_init = cv.take<float>(B * d.Sc * 16);
        p.pol_h = cv.take<float>(B * d.Sc * 16);
        p.pol_msg = cv.take<float>(B * d.Sc * 16);
        p.pol_h_dag = cv.take<float>(B * c.max_jobs * 16);
        p.pol_g = cv.take<float>(B * c.max_jobs * 16);
        p.pol_h_glob = cv.take<float>(B * 16);
        p.pol_row_start = cv.take<int32_t>(B * d.Sc);
        p.pol_stage_logits = cv.take<float>(B * d.Sc);
        p.pol_exec_logits = cv.take<float>(B * p.Epad);
        p.pol_action = cv.take<int32_t>(B * 4);
        p.pol_lgprob = cv.take<float>(B);
        p.pol_entropy = cv.take<float>(B);
        {   // scratch that parks the live observation during ssb_decima_evaluate (same layout as a snapshot)
            size_t sb = 0;
            const size_t parts[8] = {B * sizeof(ssb_obs_hdr), B * d.Mc * 2 * sizeof(int32_t),
                                     B * (c.max_jobs + 1) * sizeof(int32_t), B * d.Sc * 5 * sizeof(float), B * d.Sc,
                                     B * c.max_jobs * sizeof(int32_t), B * d.Mc * sizeof(uint64_t), B * sizeof(int32_t)};
            for (size_t x : parts) sb += (x + 255) & ~size_t(255);
            p.pol_snap = cv.take<char>(sb);
        }
        p.traj_d = cv.take<int32_t>(4);
        p.pol_act_a = cv.take<int32_t>(B);
        p.pol_act_n = cv.take<int32_t>(B);
        p.pl_all = cv.take<int32_t>(B * d.Sc);
        p.pl_sink = cv.take<int32_t>(B * d.Sc);
        p.pl_cand = cv.take<int32_t>(B * d.Sc);
        p.pl_cand_job = cv.take<int32_t>(B * d.Sc);
        p.pl_cand_out = cv.take<int32_t>(B * d.Sc);
        p.pl_jobs = cv.take<int32_t>(B * c.max_jobs);
        p.pl_exec = cv.take<int32_t>(B * p.Epad);
        // every masked edge contributes at most one sender and one receiver entry per level it is masked at
        p.lvl_cap = (int)std::min<size_t>(4 * B * d.Mc, (size_t)0x7fffffff);
        p.pl_lvl = cv.take<int32_t>((size_t)p.lvl_cap);
        p.pl_cnt = cv.take<int32_t>(tc::CNT_TOTAL);
        p.pl_ncand = cv.take<int32_t>(B);
        p.pl_bits = cv.take<unsigned long long>(B * d.Sc * 2);
        p.pol_wblob3 = cv.take<uint32_t>(fz::BLOB_TOTAL);
        p.pol_cand_rank = cv.take<int32_t>(B * d.Sc);
        p.fz_cursor = cv.take<int32_t>(4);
        p.as_elapsed = cv.take<double>(B);
        p.as_wall0 = cv.take<double>(B);
        p.as_rows = cv.take<int32_t>(B);
        p.as_kind = cv.take<uint8_t>(B);
        p.as_fresh = cv.take<uint8_t>(B);
        p.as_any = cv.take<int32_t>(4);
        *pol_streams = cv.take<uint32_t>(B);
    }
}

template <int ST>
static int launch_mlp_rows(ssb_env *env, const float *x, int n, float *out, cudaStream_t s)
{
    const size_t smem = sizeof(uint32_t) * fz::Blob<ST>::WORDS;
    CUDA_TRY(cudaFuncSetAttribute(fz::k_mlp_rows<ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int tiles = (n + 127) / 128;
    fz::k_mlp_rows<ST><<<std::min(tiles, env->num_sms * 4), 128, smem, s>>>(env->p.pol_wblob3, x, n, out);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, s);
    return SSB_OK;
}

struct BackwardScratch { float *gs, *ge, *d_hdag, *d_hglob, *d_hinit, *d_msg, *x_save; size_t save_rows, floats; };
BackwardScratch backward_scratch(const Params &p, float *base)
{
    BackwardScratch b{};
    size_t off = 0;
    auto take = [&](size_t n) { float *q = base ? base + off : nullptr; off += (n + 63) & ~size_t(63); return q; };
    b.gs = take((size_t)p.B * p.Sc);
    b.ge = take((size_t)p.B * p.Epad);
    b.d_hdag = take((size_t)p.B * p.Jc * 16);
    b.d_hglob = take((size_t)p.B * 16);
    b.d_hinit = take((size_t)p.B * p.Sc * 16);
    b.d_msg = take((size_t)p.B * p.Sc * 16);
    // the message-passing levels' input rows, saved while the forward pass is replayed once (k_save_rows): room for
    // three rows per node slot; a batch whose level lists are longer falls back to recomputing the levels
    b.save_rows = std::min<size_t>((size_t)p.lvl_cap, (size_t)3 * p.B * p.Sc);
    b.x_save = take(b.save_rows * 16);
    b.floats = off;
    return b;
}
int launch_mlp_backward(int stage, ssb_env *env, const int32_t *list, const int32_t *offset, const int32_t *count,
                        int level, const float *g_out, float *dW, const bwd::Bufs &bw, cudaStream_t s,
                        const float *x_in = nullptr);
template <int ST>
int launch_tile(ssb_env *env, const int32_t *list, const int32_t *offset, const int32_t *count, int level,
                cudaStream_t s, float *x_save = nullptr, size_t x_cap = 0)
{
    tc::TileArgs a{list, offset, count, level};
    a.x_save = x_save;
    a.x_cap = (int)std::min<size_t>(x_cap, 0x7fffffff);
    fz::k_tile3<ST><<<env->num_sms * fz::tile3_ctas<ST>(), 128, sizeof(uint32_t) * fz::Blob<ST>::WORDS, s>>>(env->p, a);
    CUDA_TRY(cudaGetLastError());
    return SSB_OK;
}
template <int ST>
int prepare_tile_kernel()
{
    CUDA_TRY(cudaFuncSetAttribute(fz::k_tile3<ST>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(sizeof(uint32_t) * fz::Blob<ST>::WORDS)));
    return SSB_OK;
}

int launch_mlp_backward(int stage, ssb_env *env, const int32_t *list, const int32_t *offset, const int32_t *count,
                        int level, const float *g_out, float *dW, const bwd::Bufs &bw, cudaStream_t s, const float *x_in)
{
    CUDA_TRY(bwd::mlp_backward(stage, env->p, env->num_sms, list, offset, count, level, g_out, nullptr, nullptr, dW, bw,
                               true, x_in, s));
    return SSB_OK;
}


int ssb_i_decima_obs(ssb_env *env, cudaStream_t s)
{
    k_decima_obs_cta<<<env->p.B, ADAPTER_WARPS * 32, (sizeof(Sim::AdJob) + sizeof(int32_t)) * env->p.Jc, s>>>(env->p);
    CUDA_TRY(cudaGetLastError());
    return SSB_OK;
}

// The captured graph of ssb_rollout_decima holds Params and the auto-reset arguments BY VALUE: every setter that
// changes one of them drops the graph, the next rollout call captures it again.
void ssb_i_drop_decision_graph(ssb_env *env)
{
    if (env->dg_exec) { cudaGraphExecDestroy(env->dg_exec); env->dg_exec = nullptr; }
}


int ssb_i_policy_init(ssb_env *env)
{
    const ssb_config *cfg = &env->cfg;
    const Dims &d = env->dims;
    Params &p = env->p;
    (void)p;
    CUDA_TRY(cudaMemset(env->pol_streams, 0, sizeof(uint32_t) * (size_t)cfg->num_envs));  // stream 0 for every env
    {
        env->policy_mode = cfg->num_envs <= 2 * env->num_sms ? POLICY_FUSED : POLICY_TILES;
        if (const char *pm = getenv("SSB_DECIMA_MODE")) {  // A/B override: 0 or 1; anything else keeps the default
            if (!strcmp(pm, "0")) env->policy_mode = POLICY_TILES;
            else if (!strcmp(pm, "1")) env->policy_mode = POLICY_FUSED;
        }
        CUDA_TRY(cudaFuncSetAttribute(fz::fused::k_decima_fused, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)fz::fused::Smem::BYTES));
        {   // group size: one round of groups over the resident CTAs (two per SM) when that needs at most GMAX
            // environments per group; otherwise ~3000 observation nodes per group (full 128-row tiles within a
            // level), the group count rounded to whole rounds
            const int ctas = 2 * env->num_sms, B = cfg->num_envs;
            int G = (B + ctas - 1) / ctas;
            if (G > fz::fused::GMAX) {
                const int by_nodes = std::max(1, std::min(fz::fused::GMAX, 3072 / std::max(64, d.Sc / 4)));
                const int rounds = (B + by_nodes * ctas - 1) / (by_nodes * ctas);
                G = (B + rounds * ctas - 1) / (rounds * ctas);
            }
            G = std::max(1, std::min(G, fz::fused::GMAX));
            if (const char *fg = getenv("SSB_FUSED_GROUP")) G = std::max(1, std::min(atoi(fg), fz::fused::GMAX));
            env->fused_group = G;
        }
        int rc;
        if ((rc = prepare_tile_kernel<tc::ST_PREP>()) || (rc = prepare_tile_kernel<tc::ST_SINK>()) ||
            (rc = prepare_tile_kernel<tc::ST_MSG>()) || (rc = prepare_tile_kernel<tc::ST_RCV>()) ||
            (rc = prepare_tile_kernel<tc::ST_DAG>()) || (rc = prepare_tile_kernel<tc::ST_GLOB>()) ||
            (rc = prepare_tile_kernel<tc::ST_STAGE>()) || (rc = prepare_tile_kernel<tc::ST_EXEC>()))
            return rc;
    }
    return SSB_OK;
}

extern "C" {

int ssb_set_decima_weights(ssb_env *env, const float *weights, int32_t n_floats)
{
    if (!env || !weights || !env->p.pol_w || n_floats != dw::TOTAL) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    // state_dict order ([out][in] per Linear) -> device layout (transposed, 4-float padded; ssb_decima.cuh)
    static const int dims[7][4] = {{5, 32, 16, 16},  {16, 32, 16, 16}, {16, 32, 16, 16}, {21, 32, 16, 16},
                                   {16, 32, 16, 16}, {53, 64, 64, 1},  {36, 64, 64, 1}};
    std::vector<float> dev(dd::TOTAL, 0.0f);
    size_t src = 0, dst = 0;
    for (int m = 0; m < 7; m++) {
        for (int l = 0; l < 3; l++) {
            const int in = dims[m][l], out = dims[m][l + 1];
            for (int o = 0; o < out; o++)
                for (int i = 0; i < in; i++) dev[dst + (size_t)i * out + o] = weights[src + (size_t)o * in + i];
            src += (size_t)in * out;
            dst += dd::pad4(in * out);
            for (int o = 0; o < out; o++) dev[dst + o] = weights[src + o];
            src += out;
            dst += dd::pad4(out);
        }
    }
    if (src != (size_t)dw::TOTAL || dst != (size_t)dd::TOTAL) return SSB_E_INVALID;
    CUDA_TRY(cudaMemcpy(env->p.pol_w, dev.data(), sizeof(float) * dd::TOTAL, cudaMemcpyHostToDevice));
    // tensor-core path: per-stage blobs (canonical UMMA tiles, bf16 three-term split, biases); padding stays zero
    CUDA_TRY(cudaMemset(env->p.pol_wblob3, 0, sizeof(uint32_t) * fz::BLOB_TOTAL));
    fz::k_build_blob<tc::ST_PREP><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_SINK><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_MSG><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_RCV><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_DAG><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_GLOB><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_STAGE><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    fz::k_build_blob<tc::ST_EXEC><<<1, 128>>>(env->p.pol_w, env->p.pol_wblob3);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    return SSB_OK;
}

// The backward pass and ssb_decima_work walk the row lists of the list-driven path; the fused forward kernel does not
// build them, so they are (re)built here from the observation, the adapter's outputs and the stored action.
__global__ void __launch_bounds__(128) k_plan_exec(Params p)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const int job_idx = p.pol_action[(size_t)b * 4 + 1];
    const int cap = job_idx >= 0 ? p.dec_caps[(size_t)b * p.Jc + job_idx] : 0;
    int base = 0;
    if (lane == 0 && cap > 0) base = atomicAdd(&p.pl_cnt[tc::CNT_EXEC], cap);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (int c = lane; c < cap; c += 32) p.pl_exec[base + c] = b * p.Epad + c;
}
static int replan(ssb_env *env, cudaStream_t s)
{
    if (env->policy_mode != POLICY_FUSED) return SSB_OK;  // the list-driven forward pass left its lists in place
    const Params &p = env->p;
    const int warp_grid = (p.B + 3) / 4;
    CUDA_TRY(cudaMemsetAsync(p.pl_cnt, 0, sizeof(int32_t) * tc::CNT_TOTAL, s));
    tc::k_pol_plan_a<<<warp_grid, 128, 0, s>>>(p);
    tc::k_pol_plan_scan<<<1, 32, 0, s>>>(p);
    tc::k_pol_plan_b<<<warp_grid, 128, 0, s>>>(p);
    k_plan_exec<<<warp_grid, 128, 0, s>>>(p);
    CUDA_TRY(cudaGetLastError());
    return SSB_OK;
}

// run_adapter = false: the adapter's outputs are already in place (restored from a snapshot);
// advance_draws = false: the Philox policy stream of the envs is left where it is (pure evaluation)
static int decima_policy_impl(ssb_env *env, const int32_t *forced_stage, const int32_t *forced_num_exec,
                              int32_t *stage_idx_out, int32_t *num_exec_out, bool run_adapter, bool advance_draws,
                              cudaStream_t s, const uint8_t *active = nullptr, bool save_levels = false)
{
    Params p = env->p;
    p.pol_active = active;
    env->bw_saved = 0;
    if (env->policy_mode == POLICY_FUSED) {
        // the whole decision of every env in one persistent kernel (ssb_decima_fused.cuh)
        CUDA_TRY(cudaMemsetAsync(p.fz_cursor, 0, sizeof(int32_t) * 4, s));
        fz::fused::Args a{forced_stage, forced_num_exec, stage_idx_out, num_exec_out, p.fz_cursor,
                          run_adapter ? 1 : 0, advance_draws ? 1 : 0, env->fused_group, env->pol_streams};
        const int groups = (p.B + env->fused_group - 1) / env->fused_group;
        fz::fused::k_decima_fused<<<std::min(groups, 2 * env->num_sms), fz::fused::THREADS, fz::fused::Smem::BYTES, s>>>(p, a);
        CUDA_TRY(cudaGetLastError());
        SSB_MARK(env, s);
        return SSB_OK;
    }
    // observation adapter -> row lists -> one tensor-core tile pass per MLP (lists: ssb_decima_tc.cuh)
    const int32_t *cnt = p.pl_cnt;
    const int warp_grid = (p.B + 3) / 4;
    int rc;
    CUDA_TRY(cudaMemsetAsync(p.pl_cnt, 0, sizeof(int32_t) * tc::CNT_TOTAL, s));
    if (run_adapter && (rc = ssb_i_decima_obs(env, s))) return rc;
    tc::k_pol_plan_a<<<warp_grid, 128, 0, s>>>(p);
    tc::k_pol_plan_scan<<<1, 32, 0, s>>>(p);
    tc::k_pol_plan_b<<<warp_grid, 128, 0, s>>>(p);
    CUDA_TRY(cudaGetLastError());
    if ((rc = launch_tile<tc::ST_PREP>(env, p.pl_all, nullptr, cnt + tc::CNT_ALL, 0, s))) return rc;
    if ((rc = launch_tile<tc::ST_SINK>(env, p.pl_sink, nullptr, cnt + tc::CNT_SINK, 0, s))) return rc;
    // (an evaluation with the backward pass's scratch attached leaves every level's input rows there)
    float *xs = nullptr;
    size_t xcap = 0;
    if (save_levels && env->bw_scratch) {
        const BackwardScratch bs = backward_scratch(p, static_cast<float *>(env->bw_scratch));
        xs = bs.x_save;
        xcap = bs.save_rows;
    }
    env->bw_saved = xs != nullptr;
    for (int k = env->dmax - 1; k >= 0; k--) {  // reversed(edge_masks) (scheduler.py:214-232)
        if ((rc = launch_tile<tc::ST_MSG>(env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * k, cnt + tc::CNT_LVL + 2 * k, k, s, xs, xcap)))
            return rc;
        if ((rc = launch_tile<tc::ST_RCV>(env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * k + 1, cnt + tc::CNT_LVL + 2 * k + 1,
                                          k, s, xs, xcap)))
            return rc;
    }
    if ((rc = launch_tile<tc::ST_DAG>(env, p.pl_all, nullptr, cnt + tc::CNT_ALL, 0, s))) return rc;
    if ((rc = launch_tile<tc::ST_GLOB>(env, p.pl_jobs, nullptr, cnt + tc::CNT_JOBS, 0, s))) return rc;
    tc::k_pol_glob_sum<<<(p.B + 7) / 8, 128, 0, s>>>(p);
    if ((rc = launch_tile<tc::ST_STAGE>(env, nullptr, nullptr, cnt + tc::CNT_CAND, 0, s))) return rc;
    tc::k_pol_sample_stage<<<warp_grid, 128, 0, s>>>(p, forced_stage, env->pol_streams);
    if ((rc = launch_tile<tc::ST_EXEC>(env, p.pl_exec, nullptr, cnt + tc::CNT_EXEC, 0, s))) return rc;
    tc::k_pol_sample_exec<<<warp_grid, 128, 0, s>>>(p, forced_num_exec, stage_idx_out, num_exec_out,
                                                    advance_draws ? 1 : 0, env->pol_streams);
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, s);
    return SSB_OK;
}

int ssb_decima_policy(ssb_env *env, const int32_t *forced_stage, const int32_t *forced_num_exec,
                      int32_t *stage_idx_out, int32_t *num_exec_out, void *stream)
{
    if (!env || !env->p.pol_w) return SSB_E_INVALID;  // needs SSB_FLAG_DECIMA_POLICY
    SSB_ON_DEVICE(env);
    return decima_policy_impl(env, forced_stage, forced_num_exec, stage_idx_out, num_exec_out, true, true,
                              (cudaStream_t)stream);
}

// ---- stored observations (RolloutBuffer.obsns) and their re-evaluation (DecimaScheduler.evaluate_actions)
namespace {
struct SnapPart { void *ptr; size_t bytes; };
int snapshot_parts(const ssb_env *env, SnapPart *out)
{
    const Params &p = env->p;
    const size_t B = p.B;
    int n = 0;
    out[n++] = {p.obs_hdr, B * sizeof(ssb_obs_hdr)};
    out[n++] = {p.obs_edges, B * p.Mc * 2 * sizeof(int32_t)};
    out[n++] = {p.obs_dag_ptr, B * (p.Jc + 1) * sizeof(int32_t)};
    out[n++] = {p.dec_feat, B * p.Sc * 5 * sizeof(float)};
    out[n++] = {p.dec_stage_mask, B * p.Sc};
    out[n++] = {p.dec_caps, B * p.Jc * sizeof(int32_t)};
    out[n++] = {p.dec_edge_bits, B * p.Mc * sizeof(uint64_t)};
    out[n++] = {p.dec_depth, B * sizeof(int32_t)};
    return n;
}
size_t snapshot_bytes(const ssb_env *env)
{
    SnapPart parts[8];
    const int n = snapshot_parts(env, parts);
    size_t total = 0;
    for (int i = 0; i < n; i++) total += (parts[i].bytes + 255) & ~size_t(255);
    return total;
}
int snapshot_copy(const ssb_env *env, char *buf, bool to_buf, cudaStream_t s)
{
    SnapPart parts[8];
    const int n = snapshot_parts(env, parts);
    size_t off = 0;
    for (int i = 0; i < n; i++) {
        if (to_buf) CUDA_TRY(cudaMemcpyAsync(buf + off, parts[i].ptr, parts[i].bytes, cudaMemcpyDeviceToDevice, s));
        else CUDA_TRY(cudaMemcpyAsync(parts[i].ptr, buf + off, parts[i].bytes, cudaMemcpyDeviceToDevice, s));
        off += (parts[i].bytes + 255) & ~size_t(255);
    }
    return SSB_OK;
}
}  // namespace

// slot i of dst <- the stored observation of sample (src_step[i], src_env[i]); only the rows in use are copied
namespace {
struct GatherParts {
    size_t off[8];      // byte offset of each part inside a snapshot block
    size_t stride[8];   // bytes per environment
};
GatherParts gather_parts(const ssb_env *env)
{
    SnapPart parts[8];
    snapshot_parts(env, parts);
    GatherParts gp;
    size_t off = 0;
    for (int q = 0; q < 8; q++) {
        gp.off[q] = off;
        gp.stride[q] = parts[q].bytes / (size_t)env->p.B;
        off += (parts[q].bytes + 255) & ~size_t(255);
    }
    return gp;
}
}  // namespace
__global__ void __launch_bounds__(128)
k_snapshot_gather(Params p, GatherParts gp, const char *src, size_t block_bytes, int num_steps, const int32_t *src_step,
                  const int32_t *src_env, char *dst)
{
    const int i = blockIdx.x, tid = threadIdx.x;
    if (i >= p.B) return;
    const int k = src_step[i], b = src_env[i];
    ssb_obs_hdr *dh = reinterpret_cast<ssb_obs_hdr *>(dst + gp.off[0]) + i;
    if (k < 0 || k >= num_steps || b < 0 || b >= p.B) {  // empty slot: an observation that takes no part
        if (tid == 0) {
            ssb_obs_hdr e = {};
            e.terminated = 1;
            *dh = e;
            reinterpret_cast<int32_t *>(dst + gp.off[7])[i] = 0;
        }
        return;
    }
    const char *blk = src + (size_t)k * block_bytes;
    const ssb_obs_hdr sh = reinterpret_cast<const ssb_obs_hdr *>(blk + gp.off[0])[b];
    if (tid == 0) {
        *dh = sh;
        reinterpret_cast<int32_t *>(dst + gp.off[7])[i] = reinterpret_cast<const int32_t *>(blk + gp.off[7])[b];
    }
    auto copy4 = [&](int part, size_t bytes) {  // 4-byte words (every part but the stage mask is int32 / f32 / u64 data)
        const uint32_t *s = reinterpret_cast<const uint32_t *>(blk + gp.off[part] + (size_t)b * gp.stride[part]);
        uint32_t *d = reinterpret_cast<uint32_t *>(dst + gp.off[part] + (size_t)i * gp.stride[part]);
        for (size_t w = tid; w < bytes / 4; w += 128) d[w] = s[w];
    };
    copy4(1, (size_t)sh.num_edges * 8);              // edge links
    copy4(2, ((size_t)sh.num_active_jobs + 1) * 4);  // dag_ptr
    copy4(3, (size_t)sh.num_nodes * 20);             // node features
    copy4(5, (size_t)sh.num_active_jobs * 4);        // commit caps
    copy4(6, (size_t)sh.num_edges * 8);              // per-edge level bits
    const uint8_t *sm = reinterpret_cast<const uint8_t *>(blk + gp.off[4] + (size_t)b * gp.stride[4]);
    uint8_t *dm = reinterpret_cast<uint8_t *>(dst + gp.off[4] + (size_t)i * gp.stride[4]);
    for (int w = tid; w < sh.num_nodes; w += 128) dm[w] = sm[w];
}

// The scatter counterpart: env b's live observation -- the one the policy call just sampled its action on -- into slot
// b of block d of the attached rollout store, and its Decima-format action into [d][b]; only the rows in use are
// copied.  d = *traj_d (ssb_rollout_decima) or as_rows[b] (ssb_rollout_decima_async).  Rows that will hold no
// transition are not written: an env outside its duration (async), and in the sync rollout what k_step is about to
// do instead of a step -- re-seed the env (auto-reset) or idle on a finished episode (k_traj_post flags both 8).
__global__ void __launch_bounds__(128)
k_snapshot_scatter(Params p, GatherParts gp, RolloutStore rs, size_t block_bytes, int async, int auto_reset)
{
    const int b = blockIdx.x, tid = threadIdx.x;
    if (b >= p.B) return;
    const ssb_obs_hdr sh = p.obs_hdr[b];
    int d;
    if (async) {
        if (p.as_kind[b] != 1) return;
        d = p.as_rows[b];
    } else {
        const EnvHdr &h = p.hdr[b];
        if ((auto_reset && !h.error && (h.done || sh.truncated)) || (h.done && h.error < 1000)) return;
        d = *p.traj_d;
    }
    if (d < 0 || d >= rs.cap) return;  // (the rollouts check their row count against the capacity up front)
    char *blk = rs.snap + (size_t)d * block_bytes;
    if (tid == 0) {
        reinterpret_cast<ssb_obs_hdr *>(blk + gp.off[0])[b] = sh;
        reinterpret_cast<int32_t *>(blk + gp.off[7])[b] = p.dec_depth[b];
        rs.stage_sel[(size_t)d * p.B + b] = p.pol_action[(size_t)b * 4];
        rs.exec_sel[(size_t)d * p.B + b] = p.pol_action[(size_t)b * 4 + 2];
    }
    auto copy4 = [&](int part, const void *src, size_t bytes) {  // 4-byte words, as k_snapshot_gather
        const uint32_t *s = reinterpret_cast<const uint32_t *>(static_cast<const char *>(src) + (size_t)b * gp.stride[part]);
        uint32_t *dw = reinterpret_cast<uint32_t *>(blk + gp.off[part] + (size_t)b * gp.stride[part]);
        for (size_t w = tid; w < bytes / 4; w += 128) dw[w] = s[w];
    };
    copy4(1, p.obs_edges, (size_t)sh.num_edges * 8);              // edge links
    copy4(2, p.obs_dag_ptr, ((size_t)sh.num_active_jobs + 1) * 4);  // dag_ptr
    copy4(3, p.dec_feat, (size_t)sh.num_nodes * 20);             // node features
    copy4(5, p.dec_caps, (size_t)sh.num_active_jobs * 4);        // commit caps
    copy4(6, p.dec_edge_bits, (size_t)sh.num_edges * 8);         // per-edge level bits
    const uint8_t *sm = p.dec_stage_mask + (size_t)b * gp.stride[4];
    uint8_t *dm = reinterpret_cast<uint8_t *>(blk + gp.off[4] + (size_t)b * gp.stride[4]);
    for (int w = tid; w < sh.num_nodes; w += 128) dm[w] = sm[w];
}
static int store_scatter(ssb_env *env, bool async, cudaStream_t s)
{
    if (!env->store.snap) return SSB_OK;
    k_snapshot_scatter<<<env->p.B, 128, 0, s>>>(env->p, gather_parts(env), env->store, snapshot_bytes(env), async ? 1 : 0,
                                               env->auto_reset);
    CUDA_TRY(cudaGetLastError());
    return SSB_OK;
}

int ssb_decima_snapshot_gather(ssb_env *env, const void *snapshots, int32_t num_steps, const int32_t *src_step,
                               const int32_t *src_env, void *dst, void *stream)
{
    if (!env || !snapshots || !src_step || !src_env || !dst || num_steps < 1 || !env->p.dec_feat) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    const Params &p = env->p;
    k_snapshot_gather<<<p.B, 128, 0, (cudaStream_t)stream>>>(p, gather_parts(env), static_cast<const char *>(snapshots), snapshot_bytes(env),
                                                             num_steps, src_step, src_env, static_cast<char *>(dst));
    CUDA_TRY(cudaGetLastError());
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_decima_head_adjoint(ssb_env *env, const float *grad_lgprob, const float *grad_entropy,
                            float *grad_stage_logits, float *grad_exec_logits, void *stream)
{
    if (!env || !env->p.pol_w || !grad_lgprob || !grad_entropy || !grad_stage_logits || !grad_exec_logits)
        return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    CUDA_TRY(bwd::head_adjoint(env->p, grad_lgprob, grad_entropy, grad_stage_logits, grad_exec_logits,
                               (cudaStream_t)stream));
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_decima_head_backward(ssb_env *env, const float *grad_stage_logits, const float *grad_exec_logits,
                             float *grad_weights, float *grad_stage_inputs, float *grad_exec_inputs,
                             float *stage_inputs, float *exec_inputs, int32_t *num_rows, void *stream)
{
    if (!env || !env->p.pol_w || !grad_stage_logits || !grad_exec_logits || !grad_weights) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    cudaStream_t s = (cudaStream_t)stream;
    const Params &p = env->p;
    {
        const int rcp = replan(env, s);
        if (rcp) return rcp;
    }
    const bwd::Bufs none{nullptr, nullptr, nullptr, nullptr, nullptr};
    CUDA_TRY(bwd::mlp_backward(tc::ST_STAGE, p, env->num_sms, nullptr, nullptr, p.pl_cnt + tc::CNT_CAND, 0,
                               grad_stage_logits, grad_stage_inputs, stage_inputs, grad_weights, none, false, nullptr, s));
    CUDA_TRY(bwd::mlp_backward(tc::ST_EXEC, p, env->num_sms, p.pl_exec, nullptr, p.pl_cnt + tc::CNT_EXEC, 0,
                               grad_exec_logits, grad_exec_inputs, exec_inputs, grad_weights, none, false, nullptr, s));
    if (num_rows) {
        int32_t c[tc::CNT_OVERFLOW + 1];
        CUDA_TRY(cudaMemcpyAsync(c, p.pl_cnt, sizeof(c), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        num_rows[0] = c[tc::CNT_CAND];
        num_rows[1] = c[tc::CNT_EXEC];
    }
    SSB_MARK(env, s);
    return SSB_OK;
}

int ssb_decima_attach_backward_scratch(ssb_env *env, void *scratch)
{
    if (!env || !env->p.pol_w || (reinterpret_cast<uintptr_t>(scratch) & 15)) return SSB_E_INVALID;
    env->bw_scratch = scratch;
    env->bw_saved = 0;
    return SSB_OK;
}

int ssb_decima_backward_bytes(ssb_env *env, size_t *bytes)
{
    if (!env || !bytes || !env->p.pol_w) return SSB_E_INVALID;
    *bytes = backward_scratch(env->p, nullptr).floats * sizeof(float);
    return SSB_OK;
}

int ssb_decima_backward(ssb_env *env, const float *grad_lgprob, const float *grad_entropy, float *grad_weights,
                        float *grad_node_embeddings, int32_t through_node_encoder, void *scratch, void *stream)
{
    if (!env || !env->p.pol_w || !grad_lgprob || !grad_entropy || !grad_weights || !grad_node_embeddings || !scratch ||
        (reinterpret_cast<uintptr_t>(scratch) & 15))
        return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    cudaStream_t s = (cudaStream_t)stream;
    const Params &p = env->p;
    const BackwardScratch b = backward_scratch(p, static_cast<float *>(scratch));
    {
        const int rcp = replan(env, s);
        if (rcp) return rcp;
    }
    CUDA_TRY(cudaMemsetAsync(grad_node_embeddings, 0, sizeof(float) * (size_t)p.B * p.Sc * 16, s));
    CUDA_TRY(cudaMemsetAsync(b.d_hdag, 0, sizeof(float) * (size_t)p.B * p.Jc * 16, s));
    CUDA_TRY(cudaMemsetAsync(b.d_hglob, 0, sizeof(float) * (size_t)p.B * 16, s));
    CUDA_TRY(bwd::head_adjoint(p, grad_lgprob, grad_entropy, b.gs, b.ge, s));
    const bwd::Bufs bw{grad_node_embeddings, b.d_hdag, b.d_hglob, b.d_hinit, b.d_msg};
    const int32_t *cnt = p.pl_cnt;
    float *gw = grad_weights;
    int rc;
    // heads first (their input gradients feed all three summaries), then the global summary, then the job summaries
    if ((rc = launch_mlp_backward(tc::ST_STAGE, env, nullptr, nullptr, cnt + tc::CNT_CAND, 0, b.gs, gw, bw, s))) return rc;
    if ((rc = launch_mlp_backward(tc::ST_EXEC, env, p.pl_exec, nullptr, cnt + tc::CNT_EXEC, 0, b.ge, gw, bw, s))) return rc;
    if ((rc = launch_mlp_backward(tc::ST_GLOB, env, p.pl_jobs, nullptr, cnt + tc::CNT_JOBS, 0, nullptr, gw, bw, s))) return rc;
    if ((rc = launch_mlp_backward(tc::ST_DAG, env, p.pl_all, nullptr, cnt + tc::CNT_ALL, 0, nullptr, gw, bw, s))) return rc;
    if (!through_node_encoder) { SSB_MARK(env, s); return SSB_OK; }
    // NodeEncoder (scheduler.py:191-234), the levels in the reverse of the forward order.  Level k's backward needs
    // the embeddings as they were BEFORE level k (the senders' inputs) and the level's aggregated messages (the
    // receivers' inputs); the forward pass overwrites both in place.  The forward level loop is therefore replayed
    // ONCE here, every level's input rows saved at their list positions (k_save_rows), and the levels' backward
    // kernels read them back -- 2 * depth tile passes.  (Round 1 recomputed reset .. level k+1 for every level k:
    // O(depth^2) passes; that path remains for batches whose level lists exceed the save area.)
    CUDA_TRY(cudaMemsetAsync(b.d_hinit, 0, sizeof(float) * (size_t)p.B * p.Sc * 16, s));
    CUDA_TRY(cudaMemsetAsync(b.d_msg, 0, sizeof(float) * (size_t)p.B * p.Sc * 16, s));
    int32_t hc[tc::CNT_TOTAL];  // the lists' lengths on the host: empty levels are skipped
    CUDA_TRY(cudaMemcpyAsync(hc, p.pl_cnt, sizeof(hc), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (hc[tc::CNT_OVERFLOW]) return SSB_E_INVALID;
    size_t lvl_rows = 0;
    int top = 0;  // number of levels in use
    for (int k = 0; k < env->dmax; k++) {
        const size_t n = (size_t)hc[tc::CNT_LVL + 2 * k] + (size_t)hc[tc::CNT_LVL + 2 * k + 1];
        if (n) top = k + 1;
        lvl_rows += n;
    }
    const bool saved = lvl_rows <= b.save_rows && !getenv("SSB_BACKWARD_RECOMPUTE");
    if (saved) {
        // the rows are already there when the evaluation this call differentiates ran with this scratch attached
        const bool have = env->bw_saved && env->bw_scratch == scratch && env->policy_mode != POLICY_FUSED;
        if (top > 0 && !have) {
            if ((rc = launch_tile<tc::ST_PREP>(env, p.pl_all, nullptr, cnt + tc::CNT_ALL, 0, s))) return rc;
            if ((rc = launch_tile<tc::ST_SINK>(env, p.pl_sink, nullptr, cnt + tc::CNT_SINK, 0, s))) return rc;
        }
        for (int j = top - 1; j >= 0 && !have; j--) {
            const int32_t *om = cnt + tc::OFF_LVL + 2 * j, *cm = cnt + tc::CNT_LVL + 2 * j;
            if ((rc = launch_tile<tc::ST_MSG>(env, p.pl_lvl, om, cm, j, s, b.x_save, b.save_rows))) return rc;
            if (j > 0) {
                if ((rc = launch_tile<tc::ST_RCV>(env, p.pl_lvl, om + 1, cm + 1, j, s, b.x_save, b.save_rows))) return rc;
            } else {
                CUDA_TRY(bwd::save_rows(tc::ST_RCV, p, env->num_sms, p.pl_lvl, om + 1, cm + 1, j, b.x_save, s));
            }
        }
        // (level 0's receive pass is not replayed: nothing reads the embeddings after it.  They are left as of
        // before level 0 -- the forward pass's outputs in pol_h are NOT restored; the heads' backward above has
        // already consumed them, and the next policy / evaluate call recomputes everything.)
        for (int k = 0; k < top; k++) {
            const int32_t *om = cnt + tc::OFF_LVL + 2 * k, *cm = cnt + tc::CNT_LVL + 2 * k;
            if ((rc = launch_mlp_backward(tc::ST_RCV, env, p.pl_lvl, om + 1, cm + 1, k, nullptr, gw, bw, s, b.x_save))) return rc;
            if ((rc = launch_mlp_backward(tc::ST_MSG, env, p.pl_lvl, om, cm, k, nullptr, gw, bw, s, b.x_save))) return rc;
        }
    } else {
        for (int k = 0; k < top; k++) {
            if ((rc = launch_tile<tc::ST_PREP>(env, p.pl_all, nullptr, cnt + tc::CNT_ALL, 0, s))) return rc;
            if ((rc = launch_tile<tc::ST_SINK>(env, p.pl_sink, nullptr, cnt + tc::CNT_SINK, 0, s))) return rc;
            for (int j = top - 1; j > k; j--) {
                if ((rc = launch_tile<tc::ST_MSG>(env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * j, cnt + tc::CNT_LVL + 2 * j, j, s)))
                    return rc;
                if ((rc = launch_tile<tc::ST_RCV>(env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * j + 1,
                                                  cnt + tc::CNT_LVL + 2 * j + 1, j, s)))
                    return rc;
            }
            if ((rc = launch_tile<tc::ST_MSG>(env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * k, cnt + tc::CNT_LVL + 2 * k, k, s)))
                return rc;
            if ((rc = launch_mlp_backward(tc::ST_RCV, env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * k + 1,
                                          cnt + tc::CNT_LVL + 2 * k + 1, k, nullptr, gw, bw, s)))
                return rc;
            if ((rc = launch_mlp_backward(tc::ST_MSG, env, p.pl_lvl, cnt + tc::OFF_LVL + 2 * k, cnt + tc::CNT_LVL + 2 * k, k,
                                          nullptr, gw, bw, s)))
                return rc;
        }
    }
    if ((rc = launch_mlp_backward(tc::ST_SINK, env, p.pl_sink, nullptr, cnt + tc::CNT_SINK, 0, nullptr, gw, bw, s))) return rc;
    if ((rc = launch_mlp_backward(tc::ST_PREP, env, p.pl_all, nullptr, cnt + tc::CNT_ALL, 0, nullptr, gw, bw, s))) return rc;
    SSB_MARK(env, s);
    return SSB_OK;
}

int ssb_decima_snapshot_bytes(ssb_env *env, size_t *bytes)
{
    if (!env || !bytes || !env->p.dec_feat) return SSB_E_INVALID;
    *bytes = snapshot_bytes(env);
    return SSB_OK;
}

int ssb_decima_snapshot(ssb_env *env, void *dst, void *stream)
{
    if (!env || !dst || !env->p.dec_feat) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    {
        const int rco = ssb_i_decima_obs(env, (cudaStream_t)stream);  // the adapter's view of the state
        if (rco) return rco;
    }
    const int rcs = snapshot_copy(env, static_cast<char *>(dst), true, (cudaStream_t)stream);
    if (rcs) return rcs;
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_decima_snapshot_load(ssb_env *env, const void *snapshot, void *stream)
{
    if (!env || !snapshot || !env->p.pol_w || env->snap_loaded) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    // the live observation is parked in the handle's scratch while the stored one is worked on
    if ((rc = snapshot_copy(env, env->p.pol_snap, true, s))) return rc;
    if ((rc = snapshot_copy(env, const_cast<char *>(static_cast<const char *>(snapshot)), false, s))) return rc;
    env->snap_loaded = 1;
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_decima_snapshot_unload(ssb_env *env, void *stream)
{
    if (!env || !env->p.pol_w || !env->snap_loaded) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    env->snap_loaded = 0;
    const int rcs = snapshot_copy(env, env->p.pol_snap, false, (cudaStream_t)stream);
    if (rcs) return rcs;
    SSB_MARK(env, stream);
    return SSB_OK;
}

int ssb_decima_evaluate(ssb_env *env, const void *snapshot, const int32_t *stage_sel, const int32_t *exec_sel,
                        float *lgprob_out, float *entropy_out, void *stream)
{
    if (!env || !stage_sel || !exec_sel || !env->p.pol_w) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    if (!snapshot && !env->snap_loaded) return SSB_E_INVALID;  // NULL: the snapshot ssb_decima_snapshot_load put in place
    cudaStream_t s = (cudaStream_t)stream;
    const size_t B = env->p.B;
    int rc;
    if (snapshot && (rc = ssb_decima_snapshot_load(env, snapshot, stream))) return rc;
    // whatever happens below, a snapshot this call loaded is unloaded again (the live observation comes back)
    rc = decima_policy_impl(env, stage_sel, exec_sel, nullptr, nullptr, false, false, s, nullptr, true);
    if (!rc && lgprob_out &&
        cudaMemcpyAsync(lgprob_out, env->p.pol_lgprob, B * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess) rc = SSB_E_CUDA;
    if (!rc && entropy_out &&
        cudaMemcpyAsync(entropy_out, env->p.pol_entropy, B * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess) rc = SSB_E_CUDA;
    if (rc == SSB_E_CUDA && !g_cuda_err[0]) snprintf(g_cuda_err, sizeof(g_cuda_err), "ssb_decima_evaluate: %s",
                                                      cudaGetErrorString(cudaGetLastError()));
    if (snapshot) {
        const int rc2 = ssb_decima_snapshot_unload(env, stream);
        if (!rc) rc = rc2;
    }
    if (!rc) SSB_MARK(env, stream);
    return rc;
}

// ---- fixed-duration Decima rollouts spanning resets (RolloutWorkerAsync.collect_rollout, rollout_worker.py:160-206)
// round = { who takes part ; policy ; row + step (or reset) ; bookkeeping }
__global__ void k_dasync_begin(Params p, double duration, int max_rows)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b == 0) *p.as_any = 0;
    if (b >= p.B) return;
    const ssb_obs_hdr &o = p.obs_hdr[b];
    int kind = 0;
    if (p.as_elapsed[b] < duration && p.as_rows[b] < max_rows && !(o.error && o.error != SSB_ENV_DONE) && !p.hdr[b].error)
        kind = (p.hdr[b].done || o.truncated) ? 2 : 1;  // the reset of :196-200, applied when the loop comes back around
    p.as_kind[b] = (uint8_t)kind;
}
__global__ void k_dasync_pre(Params p, const int32_t *a, const int32_t *n, ssb_transition *traj, int max_rows)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B || p.as_kind[b] != 1) return;
    ssb_transition t;  // rollout_buffer.add(obs, elapsed_time, action, lgprob, reward) (:191): reward filled in below
    t.wall_time = p.as_elapsed[b]; t.reward = 0.0; t.stage_idx = a[b]; t.num_exec = n[b];
    t.flags = p.as_fresh[b] ? 4 : 0;
    t.lgprob = p.pol_lgprob[b];
    traj[(size_t)b * max_rows + p.as_rows[b]] = t;
    p.as_wall0[b] = p.obs_hdr[b].wall_time;
}
__global__ void k_dasync_post(Params p, ssb_transition *traj, int max_rows, double duration)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B) return;
    const int kind = p.as_kind[b];
    if (kind == 2) { p.as_fresh[b] = 1; atomicAdd(p.as_any, 1); return; }
    if (kind != 1) return;
    const ssb_obs_hdr &o = p.obs_hdr[b];
    ssb_transition &t = traj[(size_t)b * max_rows + p.as_rows[b]];
    t.reward = o.reward;
    t.flags |= (o.terminated ? 1 : 0) | (o.truncated ? 2 : 0);
    p.as_elapsed[b] += o.wall_time - p.as_wall0[b];  // the duration of this step (:194)
    p.as_rows[b] += 1;
    p.as_fresh[b] = 0;
    if (p.as_elapsed[b] < duration && p.as_rows[b] < max_rows && !o.error) atomicAdd(p.as_any, 1);
}

__global__ void k_traj_next(Params p) { if (threadIdx.x == 0 && blockIdx.x == 0) *p.traj_d += 1; }

// one decision of ssb_rollout_decima, enqueued on s (captured into a CUDA graph by the caller)
static int decima_decision(ssb_env *env, int32_t num_decisions, int32_t max_events, ssb_transition *traj, cudaStream_t s)
{
    const Params &p = env->p;
    const int tb = (p.B + 127) / 128;
    int rc = ssb_decima_policy(env, nullptr, nullptr, p.pol_act_a, p.pol_act_n, s);
    if (rc) return rc;
    if ((rc = store_scatter(env, false, s))) return rc;
    if (traj) k_traj_pre<<<tb, 128, 0, s>>>(p, p.pol_act_a, p.pol_act_n, traj, num_decisions);
    if ((rc = ssb_step(env, p.pol_act_a, p.pol_act_n, nullptr, max_events, s))) return rc;
    if (traj) k_traj_post<<<tb, 128, 0, s>>>(p, traj, num_decisions);
    k_traj_next<<<1, 32, 0, s>>>(p);
    CUDA_TRY(cudaGetLastError());
    return SSB_OK;
}

int ssb_rollout_decima(ssb_env *env, int32_t num_decisions, int32_t max_events, ssb_transition *traj, void *stream)
{
    if (!env || !env->p.pol_w || num_decisions < 0) return SSB_E_INVALID;
    if (env->store.snap && num_decisions > env->store.cap) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    cudaStream_t caller = (cudaStream_t)stream, s = caller;
    // the legacy default stream cannot be captured: run on the handle's own stream, ordered after / before the
    // caller's stream with events
    const bool hop = caller == nullptr || caller == cudaStreamLegacy || caller == cudaStreamPerThread;
    if (hop && !env->no_graph) {
        s = env->own_stream;
        CUDA_TRY(cudaEventRecord(env->ev, caller));
        CUDA_TRY(cudaStreamWaitEvent(s, env->ev, 0));
    }
    CUDA_TRY(cudaMemsetAsync(env->p.traj_d, 0, sizeof(int32_t), s));
    // The ~50 launches of one decision are captured once into a CUDA graph and replayed: the kernels are short
    // (10-100 us) and strictly dependent, so the per-launch gaps are a visible share of a decision.
    // (SSB_NO_GRAPH=1 launches them one by one.)
    const bool same = env->dg_exec && env->dg_traj == traj && env->dg_k == num_decisions && env->dg_events == max_events &&
                      env->dg_autoreset == env->auto_reset && env->dg_seed_step == env->auto_seed_step &&
                      env->dg_store == env->store;
    if (!same && !env->no_graph) {
        if (env->dg_exec) { cudaGraphExecDestroy(env->dg_exec); env->dg_exec = nullptr; }
        cudaGraph_t g = nullptr;
        CUDA_TRY(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
        const int rc = decima_decision(env, num_decisions, max_events, traj, s);
        const cudaError_t ce = cudaStreamEndCapture(s, &g);
        if (rc || ce != cudaSuccess || !g) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            env->no_graph = 1;  // fall back to plain launches for this handle
        } else {
            const cudaError_t ie = cudaGraphInstantiate(&env->dg_exec, g, 0);
            cudaGraphDestroy(g);
            if (ie != cudaSuccess) { env->dg_exec = nullptr; env->no_graph = 1; cudaGetLastError(); }
            env->dg_traj = traj; env->dg_k = num_decisions; env->dg_events = max_events;
            env->dg_autoreset = env->auto_reset; env->dg_seed_step = env->auto_seed_step;
            env->dg_store = env->store;
        }
    }
    for (int d = 0; d < num_decisions; d++) {
        if (env->dg_exec && !env->no_graph) CUDA_TRY(cudaGraphLaunch(env->dg_exec, s));
        else {
            const int rc = decima_decision(env, num_decisions, max_events, traj, s);
            if (rc) return rc;
        }
    }
    if (s != caller) {
        CUDA_TRY(cudaEventRecord(env->ev, s));
        CUDA_TRY(cudaStreamWaitEvent(caller, env->ev, 0));
    }
    SSB_MARK(env, caller);
    return SSB_OK;
}

int ssb_decima_mlp_rows(ssb_env *env, int32_t mlp, const float *x, int32_t n_rows, float *out, void *stream)
{
    if (!env || !env->p.pol_w || !x || !out || n_rows < 1) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    cudaStream_t s = (cudaStream_t)stream;
    switch (mlp) {
    case 0: return launch_mlp_rows<tc::ST_PREP>(env, x, n_rows, out, s);
    case 1: return launch_mlp_rows<tc::ST_MSG>(env, x, n_rows, out, s);
    case 2: return launch_mlp_rows<tc::ST_RCV>(env, x, n_rows, out, s);
    case 3: return launch_mlp_rows<tc::ST_DAG>(env, x, n_rows, out, s);
    case 4: return launch_mlp_rows<tc::ST_GLOB>(env, x, n_rows, out, s);
    case 5: return launch_mlp_rows<tc::ST_STAGE>(env, x, n_rows, out, s);
    case 6: return launch_mlp_rows<tc::ST_EXEC>(env, x, n_rows, out, s);
    default: return SSB_E_INVALID;
    }
}

int ssb_decima_work(ssb_env *env, int64_t *out)
{
    if (!env || !out || !env->p.pol_w) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    CUDA_TRY(cudaDeviceSynchronize());
    {
        const int rcp = replan(env, env->own_stream);
        if (rcp) return rcp;
    }
    CUDA_TRY(cudaDeviceSynchronize());
    std::vector<int32_t> c(tc::CNT_TOTAL);
    CUDA_TRY(cudaMemcpy(c.data(), env->p.pl_cnt, sizeof(int32_t) * tc::CNT_TOTAL, cudaMemcpyDeviceToHost));
    int64_t send = 0, recv = 0;
    for (int k = 0; k < tc::MAX_LEVELS; k++) { send += c[tc::CNT_LVL + 2 * k]; recv += c[tc::CNT_LVL + 2 * k + 1]; }
    const int64_t gnn = 16 * 32 + 32 * 16 + 16 * 16;  // one 16 -> 32 -> 16 -> 16 MLP
    out[0] = c[tc::CNT_ALL]; out[1] = c[tc::CNT_SINK]; out[2] = c[tc::CNT_CAND]; out[3] = c[tc::CNT_JOBS];
    out[4] = c[tc::CNT_EXEC]; out[5] = send; out[6] = recv;
    out[7] = out[0] * ((5 * 32 + 32 * 16 + 16 * 16) + (21 * 32 + 32 * 16 + 16 * 16)) + (out[1] + send + recv + out[3]) * gnn +
             out[2] * (53 * 64 + 64 * 64 + 64) + out[4] * (36 * 64 + 64 * 64 + 64);
    return SSB_OK;
}

int ssb_rollout_decima_async(ssb_env *env, int32_t max_decisions, double rollout_duration, uint64_t seed_step,
                             ssb_transition *traj, int32_t *num_steps, double *elapsed, void *stream)
{
    if (!env || !env->p.pol_w || max_decisions < 1 || !(rollout_duration > 0.0) || !traj) return SSB_E_INVALID;
    if (env->store.snap && max_decisions > env->store.cap) return SSB_E_INVALID;
    SSB_ON_DEVICE(env);
    cudaStream_t s = (cudaStream_t)stream;
    const Params &p = env->p;
    const int tb = (p.B + 127) / 128;
    CUDA_TRY(cudaMemsetAsync(p.as_elapsed, 0, sizeof(double) * (size_t)p.B, s));
    CUDA_TRY(cudaMemsetAsync(p.as_rows, 0, sizeof(int32_t) * (size_t)p.B, s));
    CUDA_TRY(cudaMemsetAsync(p.as_fresh, 0, (size_t)p.B, s));  // (a reset round is always followed by its env's decision)
    int any = 1, rounds = 0;
    while (any) {
        // a few rounds per host check of "is any env still inside its rollout"; finished envs cost nothing in the
        // policy (treated as absent) and are masked out of the step
        for (int r = 0; r < 8; r++, rounds++) {
            k_dasync_begin<<<tb, 128, 0, s>>>(p, rollout_duration, max_decisions);
            int rc = decima_policy_impl(env, nullptr, nullptr, p.pol_act_a, p.pol_act_n, true, true, s, p.as_kind);
            if (rc) return rc;
            if ((rc = store_scatter(env, true, s))) return rc;
            k_dasync_pre<<<tb, 128, 0, s>>>(p, p.pol_act_a, p.pol_act_n, traj, max_decisions);
            // mask = as_kind (0: untouched); finished episodes are re-seeded with seed + seed_step * reset_count
            if ((rc = ssb_i_step_launch(env, p.pol_act_a, p.pol_act_n, p.as_kind, 0, nullptr, nullptr, 0, s, 1, seed_step))) return rc;
            k_dasync_post<<<tb, 128, 0, s>>>(p, traj, max_decisions, rollout_duration);
            CUDA_TRY(cudaGetLastError());
        }
        CUDA_TRY(cudaMemcpyAsync(&any, p.as_any, sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (rounds > 4 * max_decisions + 64) break;  // (every round either writes a row or resets an env)
    }
    if (num_steps) CUDA_TRY(cudaMemcpyAsync(num_steps, p.as_rows, sizeof(int32_t) * (size_t)p.B, cudaMemcpyDeviceToDevice, s));
    if (elapsed) CUDA_TRY(cudaMemcpyAsync(elapsed, p.as_elapsed, sizeof(double) * (size_t)p.B, cudaMemcpyDeviceToDevice, s));
    SSB_MARK(env, s);
    return SSB_OK;
}

int ssb_decima_attach_rollout_store(ssb_env *env, void *snapshots, int32_t capacity, int32_t *stage_sel, int32_t *exec_sel)
{
    if (!env || !env->p.pol_w) return SSB_E_INVALID;
    if (!snapshots) {
        env->store = RolloutStore{};
        return SSB_OK;
    }
    if (env->snap_loaded || capacity < 1 || !stage_sel || !exec_sel) return SSB_E_INVALID;
    env->store = RolloutStore{static_cast<char *>(snapshots), capacity, stage_sel, exec_sel};
    return SSB_OK;
}

int ssb_set_policy_streams(ssb_env *env, const uint32_t *streams)
{
    if (!env || !env->p.pol_w) return SSB_E_INVALID;
    CUDA_TRY(cudaSetDevice(env->device));
    // policy calls already enqueued sample with the streams they were enqueued with
    CUDA_TRY(cudaDeviceSynchronize());
    const size_t n = sizeof(uint32_t) * (size_t)env->p.B;
    if (streams) CUDA_TRY(cudaMemcpy(env->pol_streams, streams, n, cudaMemcpyHostToDevice));
    else CUDA_TRY(cudaMemset(env->pol_streams, 0, n));
    CUDA_TRY(cudaDeviceSynchronize());
    return SSB_OK;
}

int ssb_get_policy_views(ssb_env *env, ssb_policy_views *out)
{
    if (!env || !out || !env->p.pol_w) return SSB_E_INVALID;
    out->stage_logits = env->p.pol_stage_logits;
    out->exec_logits = env->p.pol_exec_logits;
    out->action = env->p.pol_action;
    out->lgprob = env->p.pol_lgprob;
    out->entropy = env->p.pol_entropy;
    out->node_stride = env->p.Sc;
    out->exec_stride = env->p.Epad;
    return SSB_OK;
}


}  // extern "C"
