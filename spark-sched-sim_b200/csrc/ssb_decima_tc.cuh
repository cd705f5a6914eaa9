// ssb_decima_tc.cuh -- the list-driven Decima policy pass, batched ACROSS environments: row-list planning, the gather /
// scatter of one row, sampling, the adjoint of the score heads and the CUDA-core backward kernels, plus the tcgen05 /
// mbarrier PTX wrappers that the tensor-core tile routines of ssb_decima_fused.cuh use.
//
// DecimaScheduler.schedule (schedulers/decima/scheduler.py:71-99) evaluates seven small 3-layer MLPs
// (SURVEY.md App. E).  One environment offers ~16 rows per message-passing level -- far too few for a
// 128-row UMMA tile -- so the work is organised by MLP instead of by environment: a planning pass
// turns every environment's observation into flat ROW LISTS (all nodes, sinks, the senders and
// receivers of every level, jobs, schedulable stages, executor counts), and one generic tile kernel
// runs "gather 128 rows -> Linear/act/Linear/act/Linear on the tensor cores -> scatter" over a list
// (fz::k_tile3 in ssb_decima_fused.cuh: bf16 three-term split, activations in TMEM).
// The level loop of NodeEncoder (:214-232) stays the literal sequence (deepest level first, parents
// OVERWRITE their embedding) -- it is a sequence of launches over all environments at once.
#pragma once
#include "ssb_decima.cuh"

namespace ssb {
namespace tc {

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address, leading / stride byte
// offsets (all >> 4), version 1 (Blackwell), no swizzle, base offset 0
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) |
           ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_commit(uint32_t mbar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar)
                 : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(ok)
            : "r"(mbar), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot_saddr, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_saddr), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// N (a multiple of 16) consecutive fp32 columns of this thread's TMEM lane: all loads are issued before the single wait
template <int N>
__device__ __forceinline__ void tmem_ld_row(uint32_t taddr, float *v)
{
    uint32_t r[N];
#pragma unroll
    for (int c = 0; c < N; c += 16)
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
            "[%16];"
            : "=r"(r[c + 0]), "=r"(r[c + 1]), "=r"(r[c + 2]), "=r"(r[c + 3]), "=r"(r[c + 4]), "=r"(r[c + 5]),
              "=r"(r[c + 6]), "=r"(r[c + 7]), "=r"(r[c + 8]), "=r"(r[c + 9]), "=r"(r[c + 10]), "=r"(r[c + 11]),
              "=r"(r[c + 12]), "=r"(r[c + 13]), "=r"(r[c + 14]), "=r"(r[c + 15])
            : "r"(taddr + c)
            : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < N; i++) v[i] = __uint_as_float(r[i]);
}

// ------------------------------------------------------------------ row lists and counters
// p.pl_cnt layout (int32): list lengths, then per level k: senders at [CNT_LVL + 2k], receivers at
// [CNT_LVL + 2k + 1]; OFF_LVL: exclusive offsets of those 128 lists into p.pl_lvl; CUR_LVL: fill cursors.
constexpr int CNT_ALL = 0, CNT_SINK = 1, CNT_CAND = 2, CNT_JOBS = 3, CNT_EXEC = 4, CNT_OVERFLOW = 5;
constexpr int MAX_LEVELS = 64;
constexpr int CNT_LVL = 8, OFF_LVL = CNT_LVL + 2 * MAX_LEVELS, CUR_LVL = OFF_LVL + 2 * MAX_LEVELS + 1;
constexpr int CNT_TOTAL = CUR_LVL + 2 * MAX_LEVELS;

enum Stage { ST_PREP, ST_SINK, ST_MSG, ST_RCV, ST_DAG, ST_GLOB, ST_STAGE, ST_EXEC };

template <int ST> struct Spec;
//                                      padded K0, real K0, H1, H2, OUT, tanh, offset of the MLP in dd layout
template <> struct Spec<ST_PREP>  { static constexpr int K0 = 8,  IN = 5,  H1 = 32, H2 = 16, OUT = 16, W = dd::PREP;  static constexpr bool TANH = false; };
template <> struct Spec<ST_SINK>  { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::UPD;   static constexpr bool TANH = false; };
template <> struct Spec<ST_MSG>   { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::MSG;   static constexpr bool TANH = false; };
template <> struct Spec<ST_RCV>   { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::UPD;   static constexpr bool TANH = false; };
template <> struct Spec<ST_DAG>   { static constexpr int K0 = 24, IN = 21, H1 = 32, H2 = 16, OUT = 16, W = dd::DAG;   static constexpr bool TANH = false; };
template <> struct Spec<ST_GLOB>  { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::GLOB;  static constexpr bool TANH = false; };
template <> struct Spec<ST_STAGE> { static constexpr int K0 = 56, IN = 53, H1 = 64, H2 = 64, OUT = 1,  W = dd::STAGE; static constexpr bool TANH = true; };
template <> struct Spec<ST_EXEC>  { static constexpr int K0 = 40, IN = 36, H1 = 64, H2 = 64, OUT = 1,  W = dd::EXEC;  static constexpr bool TANH = true; };

struct TileArgs {
    const int32_t *list;    // row ids (base of the array)
    const int32_t *offset;  // device pointer to the list's first index in `list` (nullptr: 0)
    const int32_t *count;   // device pointer to the list length
    int level;              // ST_RCV: the message-passing level whose masked edges are aggregated
    // ST_MSG / ST_RCV, optional: the rows' gathered inputs are also stored at x_save[list position] (positions below
    // x_cap) -- what the backward pass of the level needs once the embeddings have been overwritten
    float *x_save = nullptr;
    int x_cap = 0;
};

// ------------------------------------------------------------------ gather / scatter of one row
template <int ST>
__device__ __forceinline__ void gather_row(const Params &p, const TileArgs &a, int id, float *in)
{
    using S = Spec<ST>;
#pragma unroll
    for (int i = 0; i < S::K0; i++) in[i] = 0.0f;
    if (id < 0) return;
    if constexpr (ST == ST_PREP) {
#pragma unroll
        for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)id * 5 + i];
    } else if constexpr (ST == ST_SINK) {
        ld16(p.pol_h_init + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in));
    } else if constexpr (ST == ST_MSG) {
        ld16(p.pol_h + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in));
    } else if constexpr (ST == ST_RCV) {
        // agg[u] = sum of the messages of u's children over the edges masked at this level, in edge order
        const int b = id / p.Sc, u = id - b * p.Sc;
        const int32_t *edges = p.obs_edges + (size_t)b * p.Mc * 2;
        const uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
        const int M = p.obs_hdr[b].num_edges;
        // (edges of one parent are contiguous; four at a time so that their loads overlap)
        for (int e0 = p.pol_row_start[id]; e0 < M; e0 += 4) {
            int2 uv[4];
            uint64_t bits[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int e = e0 + q < M ? e0 + q : M - 1;
                uv[q] = *reinterpret_cast<const int2 *>(edges + 2 * e);
                bits[q] = ebits[e];
            }
            bool use[4], more = true;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                more = more && e0 + q < M && uv[q].x == u;
                use[q] = more && ((bits[q] >> a.level) & 1);
            }
            float m[4][16];
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (use[q]) ld16(p.pol_msg + ((size_t)b * p.Sc + uv[q].y) * 16, m[q]);
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (use[q]) {
#pragma unroll
                    for (int i = 0; i < 16; i++) in[i] += m[q][i];
                }
            if (!more) break;
        }
    } else if constexpr (ST == ST_DAG) {
#pragma unroll
        for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)id * 5 + i];
        ld16(p.pol_h + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in + 5));
    } else if constexpr (ST == ST_GLOB) {
        // h_dag[j] = sum over the job's nodes of their dag terms (kept in pol_msg), in node order
        const int b = id / p.Jc, j = id - b * p.Jc;
        const int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
        const int n1 = dag_ptr[j + 1];
        for (int n0 = dag_ptr[j]; n0 < n1; n0 += 4) {  // four rows in flight, summed in node order
            float z[4][16];
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (n0 + q < n1) ld16(p.pol_msg + ((size_t)b * p.Sc + n0 + q) * 16, z[q]);
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (n0 + q < n1) {
#pragma unroll
                    for (int i = 0; i < 16; i++) in[i] += z[q][i];
                }
        }
        st16(p.pol_h_dag + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in));
    } else if constexpr (ST == ST_STAGE) {
        // id = position in the candidate list
        const int node = p.pl_cand[id], jid = p.pl_cand_job[id], b = node / p.Sc;
#pragma unroll
        for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)node * 5 + i];
        ld16(p.pol_h + (size_t)node * 16, *reinterpret_cast<float(*)[16]>(in + 5));
        ld16(p.pol_h_dag + (size_t)jid * 16, *reinterpret_cast<float(*)[16]>(in + 21));
        ld16(p.pol_h_glob + (size_t)b * 16, *reinterpret_cast<float(*)[16]>(in + 37));
    } else if constexpr (ST == ST_EXEC) {
        // id = b * Epad + c, c = candidate executor count - 1 (scheduler.py:338-385)
        const int b = id / p.Epad, c = id - b * p.Epad;
        const int job_idx = p.pol_action[(size_t)b * 4 + 1];
        const int first = p.obs_dag_ptr[(size_t)b * (p.Jc + 1) + job_idx];
#pragma unroll
        for (int i = 0; i < 3; i++) in[i] = p.dec_feat[((size_t)b * p.Sc + first) * 5 + i];
        ld16(p.pol_h_dag + ((size_t)b * p.Jc + job_idx) * 16, *reinterpret_cast<float(*)[16]>(in + 3));
        ld16(p.pol_h_glob + (size_t)b * 16, *reinterpret_cast<float(*)[16]>(in + 19));
        in[35] = __fdiv_rn((float)c, (float)p.E);  // torch.arange(E) / E in float32 (:380)
    }
}

template <int ST>
__device__ __forceinline__ void scatter_row(const Params &p, int id, const float *out)
{
    if (id < 0) return;
    if constexpr (ST == ST_PREP) {
        st16(p.pol_h_init + (size_t)id * 16, *reinterpret_cast<const float(*)[16]>(out));
        // _forward_no_mp (:236-241) when the observation has no edge masks: h = h_init.  Otherwise the reference
        // starts h at 0 (:204) -- not stored here: every node is then either a sink (no masked edge as a parent: h =
        // update(h_init), the SINK pass) or a receiver at one level at least (h = h_init + update(agg)), and both
        // passes write h before anything reads it (a level's senders were written by the sink pass or a deeper level).
        if (p.dec_depth[id / p.Sc] == 0) st16(p.pol_h + (size_t)id * 16, *reinterpret_cast<const float(*)[16]>(out));
    } else if constexpr (ST == ST_SINK) {
        st16(p.pol_h + (size_t)id * 16, *reinterpret_cast<const float(*)[16]>(out));
    } else if constexpr (ST == ST_MSG) {
        st16(p.pol_msg + (size_t)id * 16, *reinterpret_cast<const float(*)[16]>(out));
    } else if constexpr (ST == ST_RCV) {
        float hi[16], o[16];
        ld16(p.pol_h_init + (size_t)id * 16, hi);
#pragma unroll
        for (int i = 0; i < 16; i++) o[i] = hi[i] + out[i];
        st16(p.pol_h + (size_t)id * 16, o);
    } else if constexpr (ST == ST_DAG) {
        st16(p.pol_msg + (size_t)id * 16, *reinterpret_cast<const float(*)[16]>(out));
    } else if constexpr (ST == ST_GLOB) {
        st16(p.pol_g + (size_t)id * 16, *reinterpret_cast<const float(*)[16]>(out));
    } else if constexpr (ST == ST_STAGE) {
        p.pol_stage_logits[p.pl_cand_out[id]] = out[0];
    } else if constexpr (ST == ST_EXEC) {
        p.pol_exec_logits[id] = out[0];
    }
}

template <bool TANH>
__device__ __forceinline__ float act_tc(float x)
{
    if (TANH) return tanhf(x);
    return x > 0.0f ? x : 0.2f * x;
}

// ------------------------------------------------------------------ planning kernels (one warp per env)
// Pass A: per-node level bit sets (which levels a node sends / receives at), row_start, the lists of
// all nodes / sinks / schedulable stages / jobs, and the global per-level sender / receiver counts.
__device__ inline void plan_bits_w(const Params &p, int b, int lane, int N, int M, int depth, int *hist /* smem [128] */)
{
    unsigned long long *bits = p.pl_bits + (size_t)b * p.Sc * 2;
    const int32_t *edges = p.obs_edges + (size_t)b * p.Mc * 2;
    const uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
    for (int i = lane; i < 2 * MAX_LEVELS; i += 32) hist[i] = 0;
    for (int n = lane; n < N; n += 32) { bits[2 * n] = 0ull; bits[2 * n + 1] = 0ull; }
    __syncwarp();
    if (depth > 0) {
        for (int e = lane; e < M; e += 32) {
            const int u = edges[2 * e], v = edges[2 * e + 1];
            const unsigned long long m = ebits[e];
            atomicOr(&bits[2 * v], m);      // v (child) sends at the levels of this edge
            atomicOr(&bits[2 * u + 1], m);  // u (parent) receives
            if (e == 0 || edges[2 * (e - 1)] != u) p.pol_row_start[(size_t)b * p.Sc + u] = e;  // sorted by tail
        }
    }
    __syncwarp();
    for (int n = lane; n < N; n += 32) {
        unsigned long long s = bits[2 * n], r = bits[2 * n + 1];
        while (s) { const int k = __ffsll((long long)s) - 1; s &= s - 1; atomicAdd(&hist[2 * k], 1); }
        while (r) { const int k = __ffsll((long long)r) - 1; r &= r - 1; atomicAdd(&hist[2 * k + 1], 1); }
    }
    __syncwarp();
}

#ifndef SSB_PLAN_MINB
#define SSB_PLAN_MINB 1
#endif
static __global__ void __launch_bounds__(128, SSB_PLAN_MINB) k_pol_plan_a(Params p)
{
    __shared__ int hist_s[4][2 * MAX_LEVELS];
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    int *hist = hist_s[threadIdx.x >> 5];
    const ssb_obs_hdr &oh = p.obs_hdr[b];
    const bool live = !(oh.terminated || oh.error) && (!p.pol_active || p.pol_active[b]);
    const int N = live ? oh.num_nodes : 0, M = live ? oh.num_edges : 0, Ja = live ? oh.num_active_jobs : 0;
    const int depth = live ? p.dec_depth[b] : 0;
    plan_bits_w(p, b, lane, N, M, depth, hist);
    for (int i = lane; i < 2 * depth; i += 32)
        if (hist[i]) atomicAdd(&p.pl_cnt[CNT_LVL + i], hist[i]);
    const unsigned long long *bits = p.pl_bits + (size_t)b * p.Sc * 2;
    const uint8_t *smask = p.dec_stage_mask + (size_t)b * p.Sc;
    const int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
    // reserve this env's ranges in the flat lists
    int n_sink = 0, n_cand = 0;
    for (int n0 = 0; n0 < N; n0 += 32) {
        const int n = n0 + lane;
        n_sink += __popc(__ballot_sync(FULL, n < N && depth > 0 && bits[2 * n + 1] == 0ull));
        n_cand += __popc(__ballot_sync(FULL, n < N && smask[n]));
    }
    int base_all = 0, base_sink = 0, base_cand = 0, base_jobs = 0;
    if (lane == 0) {
        base_all = atomicAdd(&p.pl_cnt[CNT_ALL], N);
        base_sink = atomicAdd(&p.pl_cnt[CNT_SINK], n_sink);
        base_cand = atomicAdd(&p.pl_cnt[CNT_CAND], n_cand);
        base_jobs = atomicAdd(&p.pl_cnt[CNT_JOBS], Ja);
        p.pl_ncand[b] = n_cand;
    }
    base_all = __shfl_sync(FULL, base_all, 0); base_sink = __shfl_sync(FULL, base_sink, 0);
    base_cand = __shfl_sync(FULL, base_cand, 0); base_jobs = __shfl_sync(FULL, base_jobs, 0);
    int cs = 0, cc = 0;
    for (int n0 = 0; n0 < N; n0 += 32) {
        const int n = n0 + lane;
        const bool is_sink = n < N && depth > 0 && bits[2 * n + 1] == 0ull, is_cand = n < N && smask[n];
        const unsigned ms = __ballot_sync(FULL, is_sink), mc = __ballot_sync(FULL, is_cand);
        const unsigned below = (1u << lane) - 1;
        if (n < N) p.pl_all[base_all + n] = b * p.Sc + n;
        if (is_sink) p.pl_sink[base_sink + cs + __popc(ms & below)] = b * p.Sc + n;
        if (is_cand) {
            int lo = 0, hi = Ja;  // job of node n: last j with dag_ptr[j] <= n
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (dag_ptr[mid] <= n) lo = mid; else hi = mid; }
            const int r = cc + __popc(mc & below);
            p.pl_cand[base_cand + r] = b * p.Sc + n;
            p.pl_cand_job[base_cand + r] = b * p.Jc + lo;
            p.pl_cand_out[base_cand + r] = b * p.Sc + r;
        }
        cs += __popc(ms); cc += __popc(mc);
    }
    for (int j = lane; j < Ja; j += 32) p.pl_jobs[base_jobs + j] = b * p.Jc + j;
}

// exclusive scan of the 2 * MAX_LEVELS level-list lengths; cursors start at the offsets
static __global__ void k_pol_plan_scan(Params p)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int run = 0;
    for (int i = 0; i < 2 * MAX_LEVELS; i++) {
        p.pl_cnt[OFF_LVL + i] = run;
        p.pl_cnt[CUR_LVL + i] = run;
        run += p.pl_cnt[CNT_LVL + i];
    }
    p.pl_cnt[OFF_LVL + 2 * MAX_LEVELS] = run;
    if (run > p.lvl_cap) p.pl_cnt[CNT_OVERFLOW] = 1;
}

// Pass B: fill the per-level sender / receiver lists
static __global__ void __launch_bounds__(128, SSB_PLAN_MINB) k_pol_plan_b(Params p)
{
    __shared__ int hist_s[4][2 * MAX_LEVELS];
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    if (p.pl_cnt[CNT_OVERFLOW]) return;
    int *hist = hist_s[threadIdx.x >> 5];
    const ssb_obs_hdr &oh = p.obs_hdr[b];
    const bool live = !(oh.terminated || oh.error) && (!p.pol_active || p.pol_active[b]);
    const int N = live ? oh.num_nodes : 0, depth = live ? p.dec_depth[b] : 0;
    if (depth == 0) return;
    const unsigned long long *bits = p.pl_bits + (size_t)b * p.Sc * 2;
    // this env's per-level counts again, then one reservation per non-empty list
    for (int i = lane; i < 2 * MAX_LEVELS; i += 32) hist[i] = 0;
    __syncwarp();
    for (int n = lane; n < N; n += 32) {
        unsigned long long s = bits[2 * n], r = bits[2 * n + 1];
        while (s) { const int k = __ffsll((long long)s) - 1; s &= s - 1; atomicAdd(&hist[2 * k], 1); }
        while (r) { const int k = __ffsll((long long)r) - 1; r &= r - 1; atomicAdd(&hist[2 * k + 1], 1); }
    }
    __syncwarp();
    for (int i = lane; i < 2 * depth; i += 32) {
        const int c = hist[i];
        hist[i] = c ? atomicAdd(&p.pl_cnt[CUR_LVL + i], c) : 0;  // becomes this env's write cursor
    }
    __syncwarp();
    for (int n = lane; n < N; n += 32) {
        unsigned long long s = bits[2 * n], r = bits[2 * n + 1];
        while (s) { const int k = __ffsll((long long)s) - 1; s &= s - 1; p.pl_lvl[atomicAdd(&hist[2 * k], 1)] = b * p.Sc + n; }
        while (r) { const int k = __ffsll((long long)r) - 1; r &= r - 1; p.pl_lvl[atomicAdd(&hist[2 * k + 1], 1)] = b * p.Sc + n; }
    }
}

// h_glob = sum over the active jobs of the global MLP's outputs (:265-276), in job order
static __global__ void __launch_bounds__(128) k_pol_glob_sum(Params p)
{
    const int b = blockIdx.x * 8 + (threadIdx.x >> 4), c = threadIdx.x & 15;
    if (b >= p.B) return;
    const ssb_obs_hdr &oh = p.obs_hdr[b];
    const int Ja = (oh.terminated || oh.error || (p.pol_active && !p.pol_active[b])) ? 0 : oh.num_active_jobs;
    float s = 0.0f;
    for (int j = 0; j < Ja; j++) s += p.pol_g[((size_t)b * p.Jc + j) * 16 + c];
    p.pol_h_glob[(size_t)b * 16 + c] = s;
}

// stage sampling (utils.sample, decima/utils.py:19-23) + the rows of the executor-count head
// streams: DEVICE u32[B], each env's policy sampling stream (ssb_set_policy_streams), the Philox counter's second word
static __global__ void __launch_bounds__(128)
k_pol_sample_stage(Params p, const int32_t *forced_stage, const uint32_t *streams)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const ssb_obs_hdr &oh = p.obs_hdr[b];
    const bool live = !(oh.terminated || oh.error) && (!p.pol_active || p.pol_active[b]);
    const int N = live ? oh.num_nodes : 0, Ja = live ? oh.num_active_jobs : 0;
    const int n_cand = live ? p.pl_ncand[b] : 0;
    const EnvHdr &h = p.hdr[b];
    const uint4 rw = philox4x32_10(h.policy_draws, streams[b], 4u, 0u, (uint32_t)h.seed, (uint32_t)(h.seed >> 32));
    const float u1 = ((float)(rw.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
    float lgprob = 0.0f, h_stage = 0.0f;
    const int stage_idx = n_cand > 0 ? sample_w(p.pol_stage_logits + (size_t)b * p.Sc, n_cand,
                                                forced_stage ? forced_stage[b] : -1, u1, lane, lgprob, &h_stage) : -1;
    int job_idx = -1, cap = 0;
    if (stage_idx >= 0 && stage_idx < n_cand) {
        const uint8_t *smask = p.dec_stage_mask + (size_t)b * p.Sc;
        const int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
        int seen = 0, node = -1;
        for (int n0 = 0; n0 < N && node < 0; n0 += 32) {
            const int n = n0 + lane;
            const unsigned bm = __ballot_sync(FULL, n < N && smask[n]);
            const int c = __popc(bm);
            if (stage_idx < seen + c) {
                unsigned m = bm;
                for (int q = stage_idx - seen; q > 0; q--) m &= m - 1;
                node = n0 + __ffs(m) - 1;
            }
            seen += c;
        }
        int lo = 0, hi = Ja;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (dag_ptr[mid] <= node) lo = mid; else hi = mid; }
        job_idx = lo;
        cap = p.dec_caps[(size_t)b * p.Jc + job_idx];
    }
    int base = 0;
    if (lane == 0) {
        int32_t *act = p.pol_action + (size_t)b * 4;
        act[0] = stage_idx; act[1] = job_idx; act[2] = 0; act[3] = n_cand;
        p.pol_lgprob[b] = lgprob;
        p.pol_entropy[b] = h_stage;  // completed by k_pol_sample_exec
        if (cap > 0) base = atomicAdd(&p.pl_cnt[CNT_EXEC], cap);
    }
    base = __shfl_sync(FULL, base, 0);
    for (int c = lane; c < cap; c += 32) p.pl_exec[base + c] = b * p.Epad + c;
}

static __global__ void __launch_bounds__(128)
k_pol_sample_exec(Params p, const int32_t *forced_num_exec, int32_t *stage_idx_out, int32_t *num_exec_out,
                  int advance_draws, const uint32_t *streams)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    EnvHdr &h = p.hdr[b];
    int32_t *act = p.pol_action + (size_t)b * 4;
    const int job_idx = act[1];
    const int cap = job_idx >= 0 ? p.dec_caps[(size_t)b * p.Jc + job_idx] : 0;
    const uint32_t pd = h.policy_draws;
    const uint4 rw = philox4x32_10(pd, streams[b], 4u, 0u, (uint32_t)h.seed, (uint32_t)(h.seed >> 32));
    const float u2 = ((float)(rw.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    float lgprob = p.pol_lgprob[b], h_exec = 0.0f;
    int num_exec = 0;
    if (cap > 0)
        num_exec = sample_w(p.pol_exec_logits + (size_t)b * p.Epad, cap, forced_num_exec ? forced_num_exec[b] : -1,
                            u2, lane, lgprob, &h_exec);
    __syncwarp();
    if (lane == 0) {
        act[2] = num_exec;
        p.pol_lgprob[b] = lgprob;
        // evaluate_actions: (stage entropy + exec entropy) / log(num_executors * nodes in the observation)
        const int N = p.obs_hdr[b].num_nodes;
        p.pol_entropy[b] = N > 0 ? (p.pol_entropy[b] + h_exec) / logf((float)(p.E * N)) : 0.0f;
        if (advance_draws && (!p.pol_active || p.pol_active[b])) h.policy_draws = pd + 1;
        if (stage_idx_out) stage_idx_out[b] = act[0];
        if (num_exec_out) num_exec_out[b] = 1 + num_exec;
    }
}

// ------------------------------------------------------------------ backward pass, first stage
// Adjoint of utils.evaluate (decima/utils.py:26-42) + the aggregation in evaluate_actions (scheduler.py:131-137):
// from d loss / d lgprob and d loss / d entropy of every env's stored action to d loss / d scores of the two heads.
//   p = softmax(z), q = clamp(p, eps, 1 - eps), lgprob = log q_a, H = -sum_j q_j log q_j
//   G_j = d loss / d p_j = g_lp [j == a] / q_a - g_H (log q_j + 1), both terms only where p_j is not clamped
//   d loss / d z_i = p_i (G_i - sum_j G_j p_j)
__device__ inline void softmax_adjoint_w(const float *z, int n, int sel, float g_lp, float g_h, int lane, float *dz)
{
    const float eps = 1.1920929e-07f;
    float mx = -INFINITY;
    for (int i = lane; i < n; i += 32) mx = fmaxf(mx, z[i]);
    for (int off = 16; off; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, off));
    float sum = 0.0f;
    for (int i = lane; i < n; i += 32) sum += expf(z[i] - mx);
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
    auto G = [&](int i, float pr) {
        const bool inside = pr >= eps && pr <= 1.0f - eps;
        if (!inside) return 0.0f;
        float g = -g_h * (logf(pr) + 1.0f);
        if (i == sel) g += g_lp / pr;
        return g;
    };
    float dot = 0.0f;
    for (int i = lane; i < n; i += 32) {
        const float pr = expf(z[i] - mx) / sum;
        dot += G(i, pr) * pr;
    }
    for (int off = 16; off; off >>= 1) dot += __shfl_xor_sync(FULL, dot, off);
    for (int i = lane; i < n; i += 32) {
        const float pr = expf(z[i] - mx) / sum;
        dz[i] = pr * (G(i, pr) - dot);
    }
}
static __global__ void __launch_bounds__(128)
k_pol_head_adjoint(Params p, const float *grad_lgprob, const float *grad_entropy, float *grad_stage, float *grad_exec)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    float *ds = grad_stage + (size_t)b * p.Sc, *de = grad_exec + (size_t)b * p.Epad;
    const int32_t *act = p.pol_action + (size_t)b * 4;
    const int n_cand = act[3], job_idx = act[1];
    const int cap = job_idx >= 0 ? p.dec_caps[(size_t)b * p.Jc + job_idx] : 0;
    const int N = p.obs_hdr[b].num_nodes;
    for (int i = lane; i < p.Sc; i += 32) ds[i] = 0.0f;
    for (int i = lane; i < p.Epad; i += 32) de[i] = 0.0f;
    if (n_cand <= 0 || N <= 0) return;
    const float g_lp = grad_lgprob[b], g_h = grad_entropy[b] / logf((float)(p.E * N));
    softmax_adjoint_w(p.pol_stage_logits + (size_t)b * p.Sc, n_cand, act[0], g_lp, g_h, lane, ds);
    if (cap > 0) softmax_adjoint_w(p.pol_exec_logits + (size_t)b * p.Epad, cap, act[2], g_lp, g_h, lane, de);
}

// ------------------------------------------------------------------ backward pass, second stage: one MLP
// Backward of one three-layer MLP over a row list (the same lists and gathers as the forward tile pass) on the CUDA
// cores in fp32.  Per 128-row tile (thread r <-> row r) the forward activations are recomputed and the deltas
// propagated with the weights read as broadcast 128-bit shared-memory loads (16 FMAs per 4 loads); everything a row
// produces -- X | A1 | A2 | D1 | D2 | D3 -- lives in ONE row-major shared-memory matrix T[128][LD], so that the
// tile's weight / bias gradients are 4 x 4 register blocks  acc += T[r][colL..+3] (x) T[r][colR..+3]  summed over the
// rows (two loads per 16 FMAs; the bias gradients use a constant (1,0,0,0) column block as their left factor).  The
// blocks are accumulated in registers over ALL tiles of the (persistent) CTA and added to the flat gradient vector
// (ABI layout of ssb_set_decima_weights) once at the end.  d loss / d input row goes to dX [rows][K0] in list
// order, the gathered input rows optionally to X_out (what a later stage needs to scatter / chain).  x_in: the
// rows' inputs as saved by k_save_rows when the forward pass ran (message-passing levels: the embeddings they
// read have been overwritten since), indexed by the row's position in p.pl_lvl.
template <int ST> struct DwOffset;
template <> struct DwOffset<ST_PREP>  { static constexpr int V = dw::PREP; };
template <> struct DwOffset<ST_SINK>  { static constexpr int V = dw::UPD; };
template <> struct DwOffset<ST_MSG>   { static constexpr int V = dw::MSG; };
template <> struct DwOffset<ST_RCV>   { static constexpr int V = dw::UPD; };
template <> struct DwOffset<ST_DAG>   { static constexpr int V = dw::DAG; };
template <> struct DwOffset<ST_GLOB>  { static constexpr int V = dw::GLOB; };
template <> struct DwOffset<ST_STAGE> { static constexpr int V = dw::STAGE; };
template <> struct DwOffset<ST_EXEC>  { static constexpr int V = dw::EXEC; };

template <int ST>
struct BwdSmem {
    using S = Spec<ST>;
    static constexpr int O4 = (S::OUT + 3) & ~3;
    // column offsets in T (floats); LD / 4 is odd, so a warp's 128-bit accesses to its own rows are conflict-free
    static constexpr int CX = 0, CA1 = CX + S::K0, CA2 = CA1 + S::H1, CD1 = CA2 + S::H2, CD2 = CD1 + S::H1;
    static constexpr int CD3 = CD2 + S::H2, CONE = CD3 + O4, COLS = CONE + 4;
    static constexpr int LD = ((COLS / 4) & 1) ? COLS : COLS + 4;
    static constexpr int W = 128 * LD;
    static constexpr int WN = dd::mlp(S::IN, S::H1, S::H2, S::OUT);
    static constexpr size_t BYTES = (size_t)(W + WN) * 4;
    // 4 x 4 gradient blocks: dW1 [K0/4][H1/4], dW2 [H1/4][H2/4], dW3 [H2/4][O4/4], then the three bias vectors
    static constexpr int N1 = (S::K0 / 4) * (S::H1 / 4), N2 = (S::H1 / 4) * (S::H2 / 4), N3 = (S::H2 / 4) * (O4 / 4);
    static constexpr int NB = (S::H1 + S::H2 + O4) / 4, NBLK = N1 + N2 + N3 + NB, PER_THREAD = (NBLK + 127) / 128;
};

template <bool TANH>
__device__ __forceinline__ float dact_tc(float a)  // derivative from the activation's OUTPUT
{
    if (TANH) return 1.0f - a * a;
    return a > 0.0f ? 1.0f : 0.2f;
}
// gradients with respect to the encoder's outputs, accumulated while the backward pass walks up the network
struct BwdBufs {
    float *d_h;      // [B][Sc][16]  node embeddings (NodeEncoder's output)
    float *d_hdag;   // [B][Jc][16]  job summaries
    float *d_hglob;  // [B][16]      global summary
    float *d_hinit;  // [B][Sc][16]  mlp_prep's output (NodeEncoder's h_init)
    float *d_msg;    // [B][Sc][16]  the current level's messages (zero between levels)
};
__device__ __forceinline__ int job_of_node(const Params &p, int b, int n)
{
    const int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
    int lo = 0, hi = p.obs_hdr[b].num_active_jobs;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (dag_ptr[mid] <= n) lo = mid; else hi = mid; }
    return lo;
}
// d loss / d output o of row (row, id)
template <int ST>
__device__ __forceinline__ float upstream(const Params &p, const float *g_out, const BwdBufs &bw, int row, int id, int o)
{
    using S = Spec<ST>;
    if (id < 0) return 0.0f;
    if constexpr (ST == ST_STAGE) return g_out[p.pl_cand_out[id]];
    else if constexpr (ST == ST_EXEC) return g_out[id];
    else if constexpr (ST == ST_GLOB) return g_out ? g_out[(size_t)row * S::OUT + o] : bw.d_hglob[(size_t)(id / p.Jc) * 16 + o];
    else if constexpr (ST == ST_DAG) {
        if (g_out) return g_out[(size_t)row * S::OUT + o];
        const int b = id / p.Sc;
        return bw.d_hdag[((size_t)b * p.Jc + job_of_node(p, b, id - b * p.Sc)) * 16 + o];
    } else if constexpr (ST == ST_RCV || ST == ST_SINK) {
        return g_out ? g_out[(size_t)row * S::OUT + o] : bw.d_h[(size_t)id * 16 + o];
    } else if constexpr (ST == ST_MSG) {
        return g_out ? g_out[(size_t)row * S::OUT + o] : bw.d_msg[(size_t)id * 16 + o];
    } else if constexpr (ST == ST_PREP) {
        if (g_out) return g_out[(size_t)row * S::OUT + o];
        // h = h_init for observations without message passing (_forward_no_mp, scheduler.py:236-241)
        return bw.d_hinit[(size_t)id * 16 + o] + (p.dec_depth[id / p.Sc] == 0 ? bw.d_h[(size_t)id * 16 + o] : 0.0f);
    } else return g_out[(size_t)row * S::OUT + o];
}
// the whole upstream row (O4 floats, zero-padded) into shared memory; 128-bit loads where the source is a 16-wide row
template <int ST>
__device__ __forceinline__ void upstream_row(const Params &p, const float *g_out, const BwdBufs &bw, int row, int id, float *dst)
{
    using S = Spec<ST>;
    constexpr int O4 = (S::OUT + 3) & ~3;
    if constexpr (S::OUT == 16 && (ST == ST_RCV || ST == ST_SINK || ST == ST_MSG || ST == ST_GLOB)) {
        float v[16];
#pragma unroll
        for (int o = 0; o < 16; o++) v[o] = 0.0f;
        if (id >= 0) {
            const float *src = g_out ? g_out + (size_t)row * 16
                             : ST == ST_MSG ? bw.d_msg + (size_t)id * 16
                             : ST == ST_GLOB ? bw.d_hglob + (size_t)(id / p.Jc) * 16 : bw.d_h + (size_t)id * 16;
            ld16(src, v);
        }
        st16(dst, v);
    } else {
#pragma unroll
        for (int o = 0; o < O4; o++) dst[o] = o < S::OUT ? upstream<ST>(p, g_out, bw, row, id, o) : 0.0f;
    }
}
// what else the row's output gradient does besides entering the MLP (delta = this row's upstream gradient)
template <int ST>
__device__ __forceinline__ void after_upstream(const Params &p, const BwdBufs &bw, int id, const float *delta, int stride)
{
    if (id < 0 || !bw.d_h) return;
    if constexpr (ST == ST_RCV) {
        // h[r] = h_init[r] + update(agg[r]) OVERWRITES h[r]: the gradient passes to h_init, nothing to the old value
        float hi[16];
        ld16(bw.d_hinit + (size_t)id * 16, hi);
#pragma unroll
        for (int o = 0; o < 16; o++) hi[o] += delta[o * stride];
        st16(bw.d_hinit + (size_t)id * 16, hi);
#pragma unroll
        for (int o = 0; o < 16; o++) hi[o] = 0.0f;
        st16(bw.d_h + (size_t)id * 16, hi);
    } else if constexpr (ST == ST_MSG) {
        float z[16];
#pragma unroll
        for (int o = 0; o < 16; o++) z[o] = 0.0f;
        st16(bw.d_msg + (size_t)id * 16, z);  // consumed: clean for the next level
    }
}
// where a row's input gradient goes (the adjoint of gather_row)
template <int ST>
__device__ __forceinline__ void consume_dx(const Params &p, const BwdBufs &bw, int id, const float *dx, int level)
{
    if (id < 0) return;
    if constexpr (ST == ST_STAGE) {
        if (!bw.d_h) return;
        const int node = p.pl_cand[id], jid = p.pl_cand_job[id], b = node / p.Sc;
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
            atomicAdd(reinterpret_cast<float4 *>(bw.d_h + (size_t)node * 16 + i), make_float4(dx[5 + i], dx[6 + i], dx[7 + i], dx[8 + i]));
            atomicAdd(reinterpret_cast<float4 *>(bw.d_hdag + (size_t)jid * 16 + i), make_float4(dx[21 + i], dx[22 + i], dx[23 + i], dx[24 + i]));
            atomicAdd(reinterpret_cast<float4 *>(bw.d_hglob + (size_t)b * 16 + i), make_float4(dx[37 + i], dx[38 + i], dx[39 + i], dx[40 + i]));
        }
    } else if constexpr (ST == ST_EXEC) {
        if (!bw.d_hdag) return;
        const int b = id / p.Epad, job_idx = p.pol_action[(size_t)b * 4 + 1];
        for (int i = 0; i < 16; i++) {
            atomicAdd(bw.d_hdag + ((size_t)b * p.Jc + job_idx) * 16 + i, dx[3 + i]);
            atomicAdd(bw.d_hglob + (size_t)b * 16 + i, dx[19 + i]);
        }
    } else if constexpr (ST == ST_GLOB) {
        if (!bw.d_hdag) return;
        for (int i = 0; i < 16; i++) atomicAdd(bw.d_hdag + (size_t)id * 16 + i, dx[i]);
    } else if constexpr (ST == ST_DAG) {
        if (!bw.d_h) return;
#pragma unroll
        for (int i = 0; i < 16; i += 4)
            atomicAdd(reinterpret_cast<float4 *>(bw.d_h + (size_t)id * 16 + i), make_float4(dx[5 + i], dx[6 + i], dx[7 + i], dx[8 + i]));
    } else if constexpr (ST == ST_RCV) {
        // agg[u] = sum of msg[v] over u's edges masked at this level: d msg[v] += d agg[u]
        if (!bw.d_msg) return;
        const int b = id / p.Sc, u = id - b * p.Sc;
        const int32_t *edges = p.obs_edges + (size_t)b * p.Mc * 2;
        const uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
        const int M = p.obs_hdr[b].num_edges;
        for (int e = p.pol_row_start[id]; e < M && edges[2 * e] == u; e++) {
            if (!((ebits[e] >> level) & 1)) continue;
            float4 *dst = reinterpret_cast<float4 *>(bw.d_msg + ((size_t)b * p.Sc + edges[2 * e + 1]) * 16);
#pragma unroll
            for (int i = 0; i < 4; i++) atomicAdd(dst + i, make_float4(dx[4 * i], dx[4 * i + 1], dx[4 * i + 2], dx[4 * i + 3]));
        }
    } else if constexpr (ST == ST_MSG) {
        if (!bw.d_h) return;
        float h[16];  // the sender's embedding before this level
        ld16(bw.d_h + (size_t)id * 16, h);
#pragma unroll
        for (int i = 0; i < 16; i++) h[i] += dx[i];
        st16(bw.d_h + (size_t)id * 16, h);
    } else if constexpr (ST == ST_SINK) {
        if (!bw.d_hinit) return;
        float h[16];
        ld16(bw.d_hinit + (size_t)id * 16, h);
#pragma unroll
        for (int i = 0; i < 16; i++) h[i] += dx[i];
        st16(bw.d_hinit + (size_t)id * 16, h);
    }
}

// one Linear + activation of the recomputed forward pass: out[o] = act(bias[o] + sum_k in[k] w[k][o]), `in` / `out` =
// this thread's row in T, w = the layer's transposed weight [K][N] in shared memory
template <int K, int CH, int N>
__device__ __forceinline__ void bwd_fwd_step(const float *in, const float *w, int k4, int o0, float (&acc)[CH])
{
    const float4 xv = *reinterpret_cast<const float4 *>(in + k4);
    const float x[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
        if (k4 + kk < K) {
#pragma unroll
            for (int c = 0; c < CH; c += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(w + (k4 + kk) * N + o0 + c);
                acc[c] = fmaf(x[kk], wv.x, acc[c]);
                acc[c + 1] = fmaf(x[kk], wv.y, acc[c + 1]);
                acc[c + 2] = fmaf(x[kk], wv.z, acc[c + 2]);
                acc[c + 3] = fmaf(x[kk], wv.w, acc[c + 3]);
            }
        }
    }
}
template <int K, int N, bool TANH>
__device__ __forceinline__ void bwd_layer_fwd(const float *in, const float *w, const float *bias, float *out)
{
    constexpr int CH = N < 16 ? N : 16, K4 = (K + 3) & ~3;
    constexpr bool SMALL = K4 * N <= 1024;  // the 16 / 32-wide GNN layers: straight-line code
#pragma unroll 1
    for (int o0 = 0; o0 < N; o0 += CH) {
        float acc[CH];
#pragma unroll
        for (int c = 0; c < CH; c++) acc[c] = bias[o0 + c];
        if constexpr (SMALL) {
#pragma unroll
            for (int k4 = 0; k4 < K4; k4 += 4) bwd_fwd_step<K, CH, N>(in, w, k4, o0, acc);
        } else {
#pragma unroll 2
            for (int k4 = 0; k4 < K4; k4 += 4) bwd_fwd_step<K, CH, N>(in, w, k4, o0, acc);
        }
#pragma unroll
        for (int c = 0; c < CH; c += 4)
            *reinterpret_cast<float4 *>(out + o0 + c) = make_float4(act_tc<TANH>(acc[c]), act_tc<TANH>(acc[c + 1]),
                                                                    act_tc<TANH>(acc[c + 2]), act_tc<TANH>(acc[c + 3]));
    }
}
// the adjoint of a Linear: s[k] = sum_o w[k][o] d[o] for k < K (d = this thread's delta row, N of them, N % 4 == 0)
template <int N>
__device__ __forceinline__ void bwd_dot4(const float *w, int k, const float (&d)[N], float (&s)[4])
{
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
        float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
        for (int o = 0; o < N; o += 4) {
            const float4 wv = *reinterpret_cast<const float4 *>(w + (k + kk) * N + o);
            a0 = fmaf(wv.x, d[o], a0);
            a1 = fmaf(wv.y, d[o + 1], a1);
            a0 = fmaf(wv.z, d[o + 2], a0);
            a1 = fmaf(wv.w, d[o + 3], a1);
        }
        s[kk] = a0 + a1;
    }
}
// delta of a hidden layer: dst[k] = dact(a[k]) * sum_o w[k][o] dout[o]  (k < K, K % 4 == 0)
template <int K, int N, bool TANH>
__device__ __forceinline__ void bwd_layer_delta(const float *dout, const float *w, const float *a, float *dst)
{
    float d[N];
#pragma unroll
    for (int o = 0; o < N; o += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(dout + o);
        d[o] = v.x; d[o + 1] = v.y; d[o + 2] = v.z; d[o + 3] = v.w;
    }
    auto step = [&](int k) {
        float s[4];
        bwd_dot4<N>(w, k, d, s);
        const float4 av = *reinterpret_cast<const float4 *>(a + k);
        *reinterpret_cast<float4 *>(dst + k) = make_float4(s[0] * dact_tc<TANH>(av.x), s[1] * dact_tc<TANH>(av.y),
                                                           s[2] * dact_tc<TANH>(av.z), s[3] * dact_tc<TANH>(av.w));
    };
    if constexpr (K * N <= 1024) {
#pragma unroll 4
        for (int k = 0; k < K; k += 4) step(k);
    } else {
#pragma unroll 2
        for (int k = 0; k < K; k += 4) step(k);
    }
}

#ifndef SSB_BWD_MINB
#define SSB_BWD_MINB 3  // three CTAs per SM fit by shared memory; stating it lets ptxas use up to 168 registers (backward 4.57 -> 4.39 ms)
#endif
template <int ST>
__global__ void __launch_bounds__(128, Spec<ST>::OUT > 1 ? SSB_BWD_MINB : 1)
k_mlp_backward(Params p, TileArgs a, const float *g_out, float *dX, float *X_out, float *dW, BwdBufs bw,
               const float *x_in)
{
    using S = Spec<ST>;
    using L = BwdSmem<ST>;
    extern __shared__ __align__(16) float bsm[];
    const int n_rows = *a.count;
    if (n_rows <= 0) return;
    const int list_off = a.offset ? *a.offset : 0;
    const int32_t *list = a.list + list_off;
    const int n_tiles = (n_rows + 127) >> 7, tid = threadIdx.x;
    if ((int)blockIdx.x >= n_tiles) return;
    float *T = bsm, *t = bsm + tid * L::LD, *W = bsm + L::W;
    for (int i = tid; i < L::WN; i += 128) W[i] = p.pol_w[S::W + i];
    // dd layout: per layer the transposed weight [in][out], then the bias, each padded to 4 floats
    const float *w1 = W, *b1 = w1 + dd::pad4(S::IN * S::H1);
    const float *w2 = W + dd::layer(S::IN, S::H1), *b2 = w2 + dd::pad4(S::H1 * S::H2);
    const float *w3 = w2 + dd::layer(S::H1, S::H2);
    *reinterpret_cast<float4 *>(t + L::CONE) = make_float4(1.0f, 0.0f, 0.0f, 0.0f);
    // this thread's gradient blocks: (left column, right column) in T
    int colL[L::PER_THREAD], colR[L::PER_THREAD];
    float acc[L::PER_THREAD][16];
#pragma unroll
    for (int j = 0; j < L::PER_THREAD; j++) {
        const int blk = tid + 128 * j;
        int cl = L::CONE, cr = L::CD3;  // (threads past the last block compute a block nobody reads)
        if (blk < L::N1) { cl = L::CX + 4 * (blk / (S::H1 / 4)); cr = L::CD1 + 4 * (blk % (S::H1 / 4)); }
        else if (blk < L::N1 + L::N2) { const int q = blk - L::N1; cl = L::CA1 + 4 * (q % (S::H1 / 4)); cr = L::CD2 + 4 * (q / (S::H1 / 4)); }
        else if (blk < L::N1 + L::N2 + L::N3) { const int q = blk - L::N1 - L::N2; cl = L::CA2 + 4 * (q % (S::H2 / 4)); cr = L::CD3 + 4 * (q / (S::H2 / 4)); }
        else if (blk < L::NBLK) cr = L::CD1 + 4 * (blk - L::N1 - L::N2 - L::N3);  // D1 | D2 | D3 are contiguous
        colL[j] = cl; colR[j] = cr;
#pragma unroll
        for (int i = 0; i < 16; i++) acc[j][i] = 0.0f;
    }
    __syncthreads();
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row = tile * 128 + tid;
        int id = -1;
        if (row < n_rows) id = (ST == ST_STAGE) ? row : list[row];
        {
            float in[S::K0];
            if (x_in && (ST == ST_MSG || ST == ST_RCV)) {
#pragma unroll
                for (int k = 0; k < S::K0; k++) in[k] = 0.0f;
                if (id >= 0) ld16(x_in + ((size_t)list_off + row) * 16, *reinterpret_cast<float(*)[16]>(in));
            } else {
                gather_row<ST>(p, a, id, in);
            }
#pragma unroll
            for (int k = 0; k < S::K0; k += 4)
                *reinterpret_cast<float4 *>(t + L::CX + k) = make_float4(in[k], in[k + 1], in[k + 2], in[k + 3]);
            if (X_out && row < n_rows) {
#pragma unroll
                for (int k = 0; k < S::K0; k++) X_out[(size_t)row * S::K0 + k] = in[k];
            }
        }
        // forward (recomputed)
        bwd_layer_fwd<S::IN, S::H1, S::TANH>(t + L::CX, w1, b1, t + L::CA1);
        bwd_layer_fwd<S::H1, S::H2, S::TANH>(t + L::CA1, w2, b2, t + L::CA2);
        // backward, this thread's row (a padding row has zero upstream gradient, hence zero deltas)
        upstream_row<ST>(p, g_out, bw, row, id, t + L::CD3);
        if (!g_out) after_upstream<ST>(p, bw, id, t + L::CD3, 1);
        if constexpr (S::OUT > 1) {
            bwd_layer_delta<S::H2, S::OUT, S::TANH>(t + L::CD3, w3, t + L::CA2, t + L::CD2);
        } else {
            const float d3 = t[L::CD3];
#pragma unroll 4
            for (int j = 0; j < S::H2; j++) t[L::CD2 + j] = w3[j] * d3 * dact_tc<S::TANH>(t[L::CA2 + j]);
        }
        bwd_layer_delta<S::H1, S::H2, S::TANH>(t + L::CD2, w2, t + L::CA1, t + L::CD1);
        if (row < n_rows) {
            float dx[S::K0], d1[S::H1];
#pragma unroll
            for (int i = 0; i < S::H1; i += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(t + L::CD1 + i);
                d1[i] = v.x; d1[i + 1] = v.y; d1[i + 2] = v.z; d1[i + 3] = v.w;
            }
#pragma unroll
            for (int k = 0; k < S::K0; k += 4) {
                float s4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                if (k + 3 < S::IN) {
                    bwd_dot4<S::H1>(w1, k, d1, s4);
                } else {
#pragma unroll
                    for (int kk = 0; kk < 4; kk++)
                        if (k + kk < S::IN) {
                            float sacc = 0.0f;
#pragma unroll
                            for (int i = 0; i < S::H1; i++) sacc = fmaf(w1[(k + kk) * S::H1 + i], d1[i], sacc);
                            s4[kk] = sacc;
                        }
                }
                dx[k] = s4[0]; dx[k + 1] = s4[1]; dx[k + 2] = s4[2]; dx[k + 3] = s4[3];
            }
            if (dX) {
#pragma unroll
                for (int k = 0; k < S::K0; k++) dX[(size_t)row * S::K0 + k] = dx[k];
            }
            consume_dx<ST>(p, bw, id, dx, a.level);
        }
        __syncthreads();
        // the tile's weight and bias gradients: this thread's blocks, summed over the 128 rows
#pragma unroll 4
        for (int r = 0; r < 128; r++) {
            const float *tr = T + r * L::LD;
#pragma unroll
            for (int j = 0; j < L::PER_THREAD; j++) {
                const float4 lv = *reinterpret_cast<const float4 *>(tr + colL[j]);
                const float4 rv = *reinterpret_cast<const float4 *>(tr + colR[j]);
                const float l4[4] = {lv.x, lv.y, lv.z, lv.w}, r4[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                for (int x = 0; x < 4; x++)
#pragma unroll
                    for (int y = 0; y < 4; y++) acc[j][4 * x + y] = fmaf(l4[x], r4[y], acc[j][4 * x + y]);
            }
        }
        __syncthreads();
    }
    // ABI layout of the MLP's gradient: W1 [H1][IN], b1, W2 [H2][H1], b2, W3 [OUT][H2], b3
    float *g = dW + DwOffset<ST>::V;
    constexpr int G_B1 = S::H1 * S::IN, G_W2 = G_B1 + S::H1, G_B2 = G_W2 + S::H2 * S::H1, G_W3 = G_B2 + S::H2,
                  G_B3 = G_W3 + S::OUT * S::H2;
#pragma unroll
    for (int j = 0; j < L::PER_THREAD; j++) {
        const int blk = tid + 128 * j;
        if (blk >= L::NBLK) continue;
        // out[x][y] -> g[base + x * sx + y * sy] for x < nx, y < ny
        int base, sx = 1, sy, nx = 4, ny = 4;
        if (blk < L::N1) {
            const int k0 = 4 * (blk / (S::H1 / 4)), i0 = 4 * (blk % (S::H1 / 4));
            base = i0 * S::IN + k0; sy = S::IN; nx = S::IN - k0;
        } else if (blk < L::N1 + L::N2) {
            const int q = blk - L::N1, i0 = 4 * (q % (S::H1 / 4)), j0 = 4 * (q / (S::H1 / 4));
            base = G_W2 + j0 * S::H1 + i0; sy = S::H1;
        } else if (blk < L::N1 + L::N2 + L::N3) {
            const int q = blk - L::N1 - L::N2, j0 = 4 * (q % (S::H2 / 4)), o0 = 4 * (q / (S::H2 / 4));
            base = G_W3 + o0 * S::H2 + j0; sy = S::H2; ny = S::OUT - o0;
        } else {
            const int c0 = 4 * (blk - L::N1 - L::N2 - L::N3);  // column of D1 | D2 | D3
            nx = 1; sy = 1;
            if (c0 < S::H1) base = G_B1 + c0;
            else if (c0 < S::H1 + S::H2) base = G_B2 + c0 - S::H1;
            else { base = G_B3 + c0 - S::H1 - S::H2; ny = S::OUT - (c0 - S::H1 - S::H2); }
        }
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
            for (int y = 0; y < 4; y++)
                if (x < nx && y < ny) atomicAdd(g + base + x * sx + y * sy, acc[j][4 * x + y]);
    }
}

// the inputs of a message-passing level's rows, kept for the backward pass (see k_mlp_backward): one thread per row
template <int ST>
__global__ void __launch_bounds__(128) k_save_rows(Params p, TileArgs a, float *x_save)
{
    static_assert(Spec<ST>::K0 == 16, "level rows are 16 wide");
    const int n_rows = *a.count;
    const int list_off = a.offset ? *a.offset : 0;
    const int32_t *list = a.list + list_off;
    for (int row = blockIdx.x * 128 + threadIdx.x; row < n_rows; row += gridDim.x * 128) {
        float in[16];
        gather_row<ST>(p, a, list[row], in);
        st16(x_save + ((size_t)list_off + row) * 16, in);
    }
}

}  // namespace tc
}  // namespace ssb
