// ssb_sim.cuh -- the scheduling loop of one environment, executed by one warp.
//
// Work split inside the warp:
//   * wide, regular work is warp-cooperative: selecting the next timeline event (arg-min over the
//     executors' pending events and the arrival cursor by shuffles), the schedulability scan over
//     active jobs, building the observation (prefix sums + ballots for compaction), the fair policy;
//   * the irregular state machine of one event (executor motion, commitments, pool membership with
//     CPython set order) runs on lane 0 while the other lanes wait at the next __syncwarp().
// Functions suffixed _w must be called by all 32 lanes with uniform arguments; all others are
// lane-0 code.  Reference citations are spark_sched_sim/spark_sched_sim.py unless another file is named.
#pragma once
#include "ssb_types.cuh"

namespace ssb {

#define FULL 0xffffffffu
// development aid: per-phase cycle counters (lane 0), compiled in only with -DSSB_PROFILE
#ifdef SSB_PROFILE
#define SSB_T0() long long t0_ = clock64()
#define SSB_TRESET() t0_ = clock64()
#define SSB_TACC(slot)                                                     \
    do {                                                                    \
        long long t1_ = clock64();                                          \
        if (lane == 0) p.prof[(size_t)b * 16 + (slot)] += (unsigned long long)(t1_ - t0_); \
        t0_ = t1_;                                                          \
    } while (0)
#define SSB_TCNT(slot, n)                                                   \
    do {                                                                    \
        if (lane == 0) p.prof[(size_t)b * 16 + (slot)] += (unsigned long long)(n); \
    } while (0)
#else
#define SSB_T0() do { } while (0)
#define SSB_TRESET() do { } while (0)
#define SSB_TACC(slot) do { } while (0)
#define SSB_TCNT(slot, n) do { } while (0)
#endif
// rarely executed state-machine pieces (executor motion, set emulation) are kept out of line so the
// hot event loop stays compact in the instruction cache
// SSB_RARE: executed a few times per episode at most (resets, table resizes, failures) -> out of line.
// SSB_COLD: the general-path state machine; measured: keeping it inline is 20 % faster than calls
// (ABI spills around every call) even though the kernel is instruction-fetch bound.
#ifndef SSB_RARE
#define SSB_RARE __noinline__
#endif
#ifndef SSB_COLD
#define SSB_COLD
#endif
#define SSB_CHK(cond)                         \
    do {                                      \
        if (!(cond)) {                        \
            fail(1000 + __LINE__);            \
            return;                           \
        }                                     \
    } while (0)
#define SSB_CHKR(cond, ret)                   \
    do {                                      \
        if (!(cond)) {                        \
            fail(1000 + __LINE__);            \
            return ret;                       \
        }                                     \
    } while (0)

// ---------------------------------------------------------------- Philox4x32-10 (Random123)
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                uint32_t k0, uint32_t k1)
{
    // (not fully unrolled on purpose: the rollout kernel is bound by instruction fetch, and the smaller
    // body measured 7 % faster end to end than the fully unrolled one -- profiles/r01_ab_unroll.txt)
#pragma unroll 2
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ uint32_t bounded(uint32_t w, uint32_t n) { return __umulhi(w, n); }

// -ln((w+1) * 2^-32) from IEEE +,-,*,/ only, never fused (oracle/philox_ref.py:neglog_u32).
__device__ __forceinline__ double neglog_u32(uint32_t w)
{
    unsigned long long k = (unsigned long long)w + 1ull;
    int e = 63 - __clzll((long long)k);
    double m = __ddiv_rn((double)k, (double)(1ull << e));
    if (m > 1.4142135623730951) { m = __dmul_rn(m, 0.5); e += 1; }
    double s = __ddiv_rn(__dadd_rn(m, -1.0), __dadd_rn(m, 1.0));
    double z = __dmul_rn(s, s);
    const double D[11] = {21.0, 19.0, 17.0, 15.0, 13.0, 11.0, 9.0, 7.0, 5.0, 3.0, 1.0};
    double p = __ddiv_rn(1.0, 23.0);
#pragma unroll
    for (int i = 0; i < 11; i++) p = __dadd_rn(__dmul_rn(p, z), __ddiv_rn(1.0, D[i]));
    double lnm = __dmul_rn(__dmul_rn(2.0, s), p);
    double el = __dmul_rn((double)(e - 32), 0.6931471805599453);
    return -__dadd_rn(lnm, el);
}

// ---------------------------------------------------------------- CPython 3.12 set look-alike
// Objects/setobject.c for small non-negative int keys (hash(i) == i); see SURVEY.md App. B.
template <typename T>
struct PSet {
    int mask, fill, used, finger;
    T *t;
    static constexpr int EMPTY = (T)~(T)0;
    static constexpr int DUMMY = (T)(~(T)0 - 1);
};

template <typename T>
__device__ SSB_COLD void ps_insert_clean(T *t, int mask, int key)  // set_insert_clean
{
    unsigned perturb = (unsigned)key, i = (unsigned)key & mask;
    for (;;) {
        if (t[i] == PSet<T>::EMPTY) { t[i] = (T)key; return; }
        if (i + 9 <= (unsigned)mask) {
#pragma unroll 1
            for (int j = 1; j <= 9; j++)
                if (t[i + j] == PSet<T>::EMPTY) { t[i + j] = (T)key; return; }
        }
        perturb >>= 5;
        i = (i * 5 + 1 + perturb) & mask;
    }
}
template <typename T>
__device__ SSB_RARE void ps_resize(PSet<T> &s, int minused, T *tmp)  // set_table_resize
{
    int newsize = 8;
    while (newsize <= minused) newsize <<= 1;
    int oldmask = s.mask;
    if (newsize == 8 && oldmask == 7 && s.fill == s.used) return;
    // (tables are at least 8 entries and 8-byte aligned: copy and fill in 64-bit words, EMPTY is all ones)
    {
        unsigned long long *t8 = reinterpret_cast<unsigned long long *>(s.t), *m8 = reinterpret_cast<unsigned long long *>(tmp);
#pragma unroll 1
        for (int i = 0; i < (oldmask + 1) * (int)sizeof(T) / 8; i++) m8[i] = t8[i];
#pragma unroll 1
        for (int i = 0; i < newsize * (int)sizeof(T) / 8; i++) t8[i] = ~0ull;
    }
    s.mask = newsize - 1;
    s.fill = s.used;
#pragma unroll 1
    for (int i = 0; i <= oldmask; i++)
        if (tmp[i] < PSet<T>::DUMMY) ps_insert_clean(s.t, s.mask, tmp[i]);
}
template <typename T>
__device__ SSB_COLD void ps_add(PSet<T> &s, int key, T *tmp)  // set_add_entry
{
    int mask = s.mask, freeslot = -1;
    unsigned perturb = (unsigned)key, i = (unsigned)key & mask;
    for (;;) {
        int probes = (i + 9 <= (unsigned)mask) ? 9 : 0;
#pragma unroll 1
        for (int j = 0; j <= probes; j++) {
            int v = s.t[i + j];
            if (v == PSet<T>::EMPTY) {
                if (freeslot >= 0) { s.used++; s.t[freeslot] = (T)key; return; }
                s.fill++; s.used++;
                s.t[i + j] = (T)key;
                if (s.fill * 5 < mask * 3) return;
                ps_resize(s, s.used * 4, tmp);
                return;
            }
            if (v == key) return;
            if (v == PSet<T>::DUMMY) freeslot = (int)(i + j);
        }
        perturb >>= 5;
        i = (i * 5 + 1 + perturb) & mask;
    }
}
template <typename T>
__device__ inline int ps_find(const PSet<T> &s, int key)  // set_lookkey
{
    int mask = s.mask;
    unsigned perturb = (unsigned)key, i = (unsigned)key & mask;
    for (;;) {
        int probes = (i + 9 <= (unsigned)mask) ? 9 : 0;
#pragma unroll 1
        for (int j = 0; j <= probes; j++) {
            int v = s.t[i + j];
            if (v == PSet<T>::EMPTY) return -1;
            if (v == key) return (int)(i + j);
        }
        perturb >>= 5;
        i = (i * 5 + 1 + perturb) & mask;
    }
}
template <typename T>
__device__ inline bool ps_remove(PSet<T> &s, int key)
{
    int slot = ps_find(s, key);
    if (slot < 0) return false;
    s.t[slot] = (T)PSet<T>::DUMMY;
    s.used--;
    return true;
}
template <typename T>
__device__ inline int ps_pop(PSet<T> &s)  // set_pop
{
    if (s.used == 0) return -1;
    int i = s.finger & s.mask;
    while (s.t[i] >= PSet<T>::DUMMY) {
        i++;
        if (i > s.mask) i = 0;
    }
    int key = s.t[i];
    s.t[i] = (T)PSet<T>::DUMMY;
    s.used--;
    s.finger = i + 1;
    return key;
}
template <typename T>
__device__ inline void ps_init(PSet<T> &s, T *table)
{
    s.mask = 7; s.fill = s.used = s.finger = 0; s.t = table;
    for (int i = 0; i < 8; i++) table[i] = (T)PSet<T>::EMPTY;
}
// set.copy(): make_new_set + set_merge into an empty set
template <typename T>
__device__ SSB_RARE void ps_copy_into(PSet<T> &dst, T *table, const PSet<T> &other, T *tmp)
{
    ps_init(dst, table);
    if (other.used == 0) return;
    if (other.used * 5 >= 7 * 3) ps_resize(dst, other.used * 2, tmp);
    if (dst.mask == other.mask && other.fill == other.used) {
        const unsigned long long *o8 = reinterpret_cast<const unsigned long long *>(other.t);
        unsigned long long *d8 = reinterpret_cast<unsigned long long *>(dst.t);
#pragma unroll 1
        for (int i = 0; i < (other.mask + 1) * (int)sizeof(T) / 8; i++) d8[i] = o8[i];
        dst.fill = other.fill; dst.used = other.used;
        return;
    }
    dst.fill = dst.used = other.used;
#pragma unroll 1
    for (int i = 0; i <= other.mask; i++)
        if (other.t[i] < PSet<T>::DUMMY) ps_insert_clean(dst.t, dst.mask, other.t[i]);
}

__device__ __forceinline__ int popc64(uint64_t x) { return __popcll(x); }
__device__ __forceinline__ int ffs64(uint64_t x) { return __ffsll((long long)x) - 1; }
__device__ __forceinline__ uint64_t bit64(int s) { return 1ull << s; }

// ================================================================ one environment, one warp
struct Sim {
    const Params &p;
    const int b, lane;
    EnvHdr *h;
    ExecRec *ex;
    JobRec *jb;
    StageRec *st;
    int16_t *act;
    Commit *cm;
    PoolHdr *ph;
    uint8_t *pt;
    uint8_t *scr;
    ssb_stats *stats;
    ssb_obs_hdr *oh;

    __device__ Sim(const Params &p_, int b_, int lane_) : p(p_), b(b_), lane(lane_)
    {
        h = p.hdr + b;
        ex = p.exec + (size_t)b * p.E;
        jb = p.job + (size_t)b * p.Jc;
        st = p.stage + (size_t)b * p.Sc;
        act = p.active + (size_t)b * p.Jc;
        cm = p.commits + (size_t)b * p.Cc;
        ph = p.pool_hdr + (size_t)b * p.P;
        pt = p.pool_tab + (size_t)b * p.P * p.TAB;
        scr = p.scr_tab + (size_t)b * 3 * p.TAB;
        stats = p.stats + b;
        oh = p.obs_hdr + b;
    }

    __device__ SSB_RARE void fail(int code)
    {
        if (!h->error) h->error = code;
    }

    // ------------------------------------------------------------ pool helpers (executor_tracker.py)
    __device__ int pool_of_job(int j) const { return 2 + j; }
    __device__ int pool_of_stage(int j, int s) const { return 2 + p.Jc + jb[j].node_base + s; }
    __device__ int pool_job(int pool) const  // pool_key[0], -1 == None
    {
        if (pool < 2) return -1;
        if (pool < 2 + p.Jc) return pool - 2;
        return st[pool - 2 - p.Jc].job;
    }
    __device__ int pool_stage(int pool) const  // pool_key[1], -1 == None
    {
        if (pool < 2 + p.Jc) return -1;
        int node = pool - 2 - p.Jc;
        return node - jb[st[node].job].node_base;
    }
    __device__ PSet<uint8_t> ps_load(int pool) const
    {
        PSet<uint8_t> s;
        PoolHdr hd = ph[pool];
        s.mask = hd.mask; s.fill = hd.fill; s.used = hd.used; s.finger = hd.finger;
        s.t = pt + (size_t)pool * p.TAB;
        return s;
    }
    __device__ void ps_store(int pool, const PSet<uint8_t> &s)
    {
        PoolHdr hd;
        hd.mask = (uint16_t)s.mask; hd.fill = (uint16_t)s.fill; hd.used = (uint16_t)s.used;
        hd.finger = (uint16_t)s.finger;
        ph[pool] = hd;
    }
    __device__ int pool_size(int pool) const { return ph[pool].used; }
    __device__ int commit_from(int pool) const
    {
        if (pool == POOL_NONE) return 0;
        if (pool == POOL_COMMON) return h->commit_from_common;
        if (pool < 2 + p.Jc) return jb[pool - 2].commit_from;
        return st[pool - 2 - p.Jc].commit_from;
    }
    __device__ void add_commit_from(int pool, int d)
    {
        if (pool == POOL_COMMON) h->commit_from_common += d;
        else if (pool < 2 + p.Jc) jb[pool - 2].commit_from += d;
        else st[pool - 2 - p.Jc].commit_from += d;
    }
    __device__ void add_total(int job, int d)  // _total_executor_count[job], job -1 == None
    {
        if (job < 0) h->total_none += d;
        else jb[job].supply += d;
    }
    // demand <= 0  (_get_executor_demand :566-578, _is_stage_saturated :580-582)
    __device__ void update_sat(int j, int s)
    {
        const StageRec &r = st[jb[j].node_base + s];
        int demand = (int)r.remaining - ((int)r.moving_to + (int)r.commit_to);
        if (demand <= 0) jb[j].sat |= bit64(s);
        else jb[j].sat &= ~bit64(s);
    }
    __device__ void add_commit_to(int pool, int d)
    {
        if (pool == POOL_COMMON) { h->commit_to_common += d; return; }
        StageRec &r = st[pool - 2 - p.Jc];
        r.commit_to += d;
        update_sat(r.job, pool_stage(pool));
    }
    __device__ int source_job_id() const  // executor_tracker.py:99-103
    {
        int s = h->source;
        if (s == POOL_NONE || s == POOL_COMMON) return -1;
        return pool_job(s);
    }
    __device__ int num_committable() const  // executor_tracker.py:105-111
    {
        int s = h->source;
        if (s == POOL_NONE) return 0;
        return (int)ph[s].used - commit_from(s);
    }
    __device__ Commit *find_commit(int src, int dst)
    {
        int n = h->n_commits;
        for (int i = 0; i < n; i++)
            if (cm[i].src == src && cm[i].dst == dst) return cm + i;
        return nullptr;
    }
    __device__ SSB_COLD void add_commitment(int n, int dst)  // executor_tracker.py:146-154, :224-236
    {
        int src = h->source;
        SSB_CHK(src != POOL_NONE);
        Commit *c = find_commit(src, dst);
        if (c) c->n += n;
        else {
            SSB_CHK(h->n_commits < p.Cc);
            Commit nc; nc.src = src; nc.dst = dst; nc.n = n;
            cm[h->n_commits++] = nc;
        }
        add_commit_from(src, n);
        add_commit_to(dst, n);
        SSB_CHK(pool_size(src) >= commit_from(src));
        int sj = pool_job(src), dj = pool_job(dst);
        if (dj != sj) add_total(dj, n);
    }
    __device__ SSB_COLD int remove_commitment(int e, int dst)  // executor_tracker.py:156-173, :238-249
    {
        int src = ex[e].loc;
        SSB_CHKR(src != POOL_NONE, POOL_NONE);
        Commit *c = find_commit(src, dst);
        SSB_CHKR(c != nullptr, POOL_NONE);
        c->n -= 1;
        add_commit_from(src, -1);
        add_commit_to(dst, -1);
        SSB_CHKR(commit_from(src) >= 0, POOL_NONE);
        if (c->n == 0) {
            int idx = (int)(c - cm), n = h->n_commits;
            for (int i = idx; i + 1 < n; i++) cm[i] = cm[i + 1];
            h->n_commits = n - 1;
        }
        int sj = pool_job(src), dj = pool_job(dst);
        if (dj != sj) {
            add_total(dj, -1);
            SSB_CHKR(dj < 0 ? h->total_none >= 0 : jb[dj].supply >= 0, POOL_NONE);
        }
        return src;
    }
    __device__ int peek_commitment(int pool)  // executor_tracker.py:175-180
    {
        int n = h->n_commits;
        for (int i = 0; i < n; i++)
            if (cm[i].src == pool) return cm[i].dst;
        return POOL_NONE;
    }
    __device__ SSB_COLD void move_executor_to_pool(int e, int new_pool, bool send)  // executor_tracker.py:186-220
    {
        int old = ex[e].loc;
        if (old != POOL_NONE) {
            PSet<uint8_t> s = ps_load(old);
            bool ok = ps_remove(s, e);
            ps_store(old, s);
            SSB_CHK(ok);
            ex[e].loc = POOL_NONE;
        }
        if (!send) {
            ex[e].loc = new_pool;
            PSet<uint8_t> s = ps_load(new_pool);
            ps_add(s, e, scr + 2 * p.TAB);
            ps_store(new_pool, s);
            return;
        }
        SSB_CHK(new_pool >= 2 + p.Jc);
        StageRec &r = st[new_pool - 2 - p.Jc];
        r.moving_to += 1;
        update_sat(r.job, pool_stage(new_pool));
        int old_job = old != POOL_NONE ? pool_job(old) : -1, new_job = r.job;
        SSB_CHK(old_job != new_job);
        jb[new_job].supply += 1;
        if (old_job != -1) {
            jb[old_job].supply -= 1;
            SSB_CHK(jb[old_job].supply >= 0);
        }
    }

    // ------------------------------------------------------------ sampler (data_samplers/tpch.py)
    __device__ bool sample_wave(int ts, int wave, int lvl, uint32_t w1, bool warmup, double &out)  // :208-214
    {
        if (lvl < 0 || !((p.b_present[ts * 4 + wave] >> lvl) & 1)) return false;  // KeyError
        uint2 oc = p.b_dur[(ts * 3 + wave) * 8 + lvl];
        if (oc.y == 0) return false;  // ValueError: choice from an empty list
        double d = p.b_vals[oc.x + bounded(w1, oc.y)];
        if (warmup) d = __dadd_rn(d, p.warmup_delay);
        out = d;
        return true;
    }
    __device__ double task_duration(int j, int s, int e)  // tpch.py:75-106
    {
        double d = 1.0;
        int rc = sample_duration(j, s, h->launch_idx, !ex[e].has_task, ex[e].task_stage == s, d);
        if (rc) fail(rc);
        return d;
    }
    // Duration of launch number `li` of the episode; `idle`: executor.task is None; `same_stage`:
    // executor.task.stage_id == stage id.  Returns 0 or an SSB_ENV_* code WITHOUT touching the
    // environment, so the batched fast path may call it speculatively from any lane.
    __device__ __forceinline__ int sample_duration(int j, int s, uint32_t li, bool idle, bool same_stage,
                                                    double &d)
    {
        return sample_duration_ts(jb[j].ts_base + s, jb[j].n_local, li, idle, same_stage, d);
    }
    // same, with the template-stage row and len(job.local_executors) already in registers
    __device__ SSB_COLD int sample_duration_ts(int ts, int n_local, uint32_t li, bool idle,
                                                bool same_stage, double &d)
    {
        if (h->use_tape) {
            if ((int)li >= h->tape_len) return SSB_ENV_TAPE_EXHAUSTED;
            d = p.tape[(size_t)b * p.tape_cap + li];
            return 0;
        }
        if (!(n_local > 0 && n_local <= p.E)) return 1000 + __LINE__;
        uint4 w = philox4x32_10(li, 0u, 2u, 0u, (uint32_t)h->seed, (uint32_t)(h->seed >> 32));
        // _sample_executor_key :216-235; iv row = (left level, right level, left index, right index)
        const short4 iv = p.iv[n_local];
        int lvl = iv.z;
        if (iv.x != iv.y) {
            double u = __dmul_rn((double)w.x, 1.0 / 4294967296.0);
            int rand_pt = 1 + (int)__dmul_rn(u, (double)(iv.y - iv.x));
            lvl = (rand_pt <= n_local - iv.x) ? iv.z : iv.w;
        }
        int fw = p.b_present[ts * 4 + 1];
        if (lvl < 0 || !((fw >> lvl) & 1)) lvl = fw ? 31 - __clz(fw) : -1;  // max(data["first_wave"])
        if (idle) {  // executor.is_idle
            if (sample_wave(ts, 0, lvl, w.y, false, d)) return 0;
            if (sample_wave(ts, 1, lvl, w.y, true, d)) return 0;
            return SSB_ENV_SAMPLER;
        }
        if (same_stage)
            if (sample_wave(ts, 2, lvl, w.y, false, d)) return 0;
        if (sample_wave(ts, 1, lvl, w.y, false, d)) return 0;
        if (sample_wave(ts, 0, lvl, w.y, false, d)) return 0;
        return SSB_ENV_SAMPLER;
    }

    // ------------------------------------------------------------ schedulability (:505-555)
    // Schedulable stages of job j as a bitmask: ready (unsaturated, all parents saturated), not yet
    // selected this round, job not saturated with executors unless it is the source job.
    __device__ SSB_COLD uint64_t job_sched_mask(int j, int source_job) const
    {
        const JobRec &J = jb[j];
        if (!(j == source_job || J.supply < p.E)) return 0;
        uint64_t sat = J.sat, cand = J.active & ~J.selected & ~sat, out = 0;
        const uint64_t *pm = p.b_parent + J.ts_base;
        while (cand) {
            int s = ffs64(cand);
            cand &= cand - 1;
            if ((pm[s] & ~sat) == 0) out |= bit64(s);
        }
        return out;
    }
    // _find_schedulable_stages over all active jobs; writes every active job's `sched` mask
    __device__ SSB_COLD int find_schedulable_all_w()
    {
        int src_job = source_job_id();
        int n_active = h->n_active, total = 0;
        for (int base = 0; base < n_active; base += 32) {
            int i = base + lane, cnt = 0;
            if (i < n_active) {
                int j = act[i];
                uint64_t m = job_sched_mask(j, src_job);
                jb[j].sched = m;
                cnt = popc64(m);
            }
            total += __reduce_add_sync(FULL, cnt);
        }
        __syncwarp();
        if (lane == 0) { h->n_sched = total; stats->sched_scans++; }
        return total;
    }
    __device__ void clear_sched_w()
    {
        int n_active = h->n_active;
        for (int i = lane; i < n_active; i += 32) jb[act[i]].sched = 0;
        if (lane == 0) h->n_sched = 0;
        __syncwarp();
    }
    // first schedulable stage of the job-id list semantics used by _find_backup_stage (:821-845)
    __device__ bool first_schedulable(bool only_job, int job, int source_job_arg, int &oj, int &os)
    {
        int src_job = source_job_arg <= 0 ? source_job_id() : source_job_arg;  // `if not source_job_id`
        if (only_job) {
            uint64_t m = job_sched_mask(job, src_job);
            if (!m) return false;
            oj = job; os = ffs64(m);
            return true;
        }
        // other_job_ids = active jobs except `job`; an EMPTY list means "all active jobs" (:518-519)
        int n_active = h->n_active;
        bool all = true;
        for (int i = 0; i < n_active; i++) if (act[i] != job) { all = false; break; }
        for (int i = 0; i < n_active; i++) {
            int j = act[i];
            if (!all && j == job) continue;
            uint64_t m = job_sched_mask(j, src_job);
            if (m) { oj = j; os = ffs64(m); return true; }
        }
        return false;
    }

    // ------------------------------------------------------------ executor motion
    // Executor.add_history (components/executor.py:34-44; read by the renderer only, spark_sched_sim.py:408-424):
    // "executor e now belongs to job (-1: the common pool) since wall_time".  Optional export, off by default.
    __device__ SSB_RARE void add_history(int e, int job)
    {
        const int n = h->hist_n;
        if (n < p.hist_cap) {
            HistRow r;
            r.t = h->wall_time; r.exec = (int16_t)e; r.job = (int16_t)job; r.pad = 0;
            p.hist[(size_t)b * p.hist_cap + n] = r;
        }
        h->hist_n = n + 1;
    }
    __device__ void detach_executor(int j, int e)  // job.py:86-89
    {
        SSB_CHK(jb[j].n_local > 0);
        jb[j].n_local -= 1;
        ex[e].job_id = -1;
        ex[e].has_task = 0;
    }
    __device__ void push_event(int e, double t, int kind, int j, int s, int task)
    {
        ExecRec &x = ex[e];
        x.ev_t = t; x.ev_seq = h->seq++; x.ev_kind = (uint8_t)kind;
        x.ev_job = (int16_t)j; x.ev_stage = (int16_t)s; x.ev_task = task;
        x.t_acc = h->wall_time;
    }
    __device__ void execute_next_task(int e, int j, int s)  // :584-615
    {
        StageRec &r = st[jb[j].node_base + s];
        SSB_CHK(r.remaining > 0);
        SSB_CHK(ex[e].job_id == j);
        SSB_CHK(!ex[e].is_executing);
        int task_id = r.remaining - 1;  // stage.py:53-58: tasks pop from the end
        r.remaining -= 1;
        if (r.remaining == 0) jb[j].sat_count += 1;
        update_sat(j, s);
        double d = task_duration(j, s, e);
        h->launch_idx += 1;
        ex[e].has_task = 1; ex[e].task_stage = (int16_t)s; ex[e].is_executing = 1;
        r.mrd = (float)d;
        push_event(e, __dadd_rn(h->wall_time, d), EV_TASK_FINISHED, j, s, task_id);
    }
    __device__ void send_executor(int e, int j, int s)  // :617-637
    {
        SSB_CHK(!ex[e].is_executing);
        SSB_CHK(ex[e].job_id != j);
        move_executor_to_pool(e, pool_of_stage(j, s), true);
        if (ex[e].job_id != -1) detach_executor(ex[e].job_id, e);
        push_event(e, __dadd_rn(h->wall_time, p.moving_delay), EV_EXECUTOR_READY, j, s, -1);
    }
    // _get_idle_source_executors (:714-728): set(generator) over a copy of the pool; result in scr[1]
    __device__ SSB_COLD PSet<uint8_t> idle_executors(int pool)
    {
        PSet<uint8_t> src = ps_load(pool), cp, idle;
        ps_copy_into(cp, scr, src, scr + 2 * p.TAB);
        ps_init(idle, scr + p.TAB);
        for (int i = 0; i <= cp.mask; i++) {
            int v = cp.t[i];
            if (v < PSet<uint8_t>::DUMMY && !ex[v].is_executing) ps_add(idle, v, scr + 2 * p.TAB);
        }
        return idle;
    }
    // _move_idle_executors (:745-782).  e >= 0: that single executor; e < 0: all idle ones at src
    __device__ SSB_COLD void move_idle_executors(int src, int e)
    {
        if (src == POOL_NONE) src = h->source;
        SSB_CHK(src != POOL_NONE);
        if (src == POOL_COMMON) return;
        uint8_t ids[128];
        int n = 0;
        if (e >= 0) ids[n++] = (uint8_t)e;
        else {
            PSet<uint8_t> idle = idle_executors(src);
            for (int i = 0; i <= idle.mask && n < 128; i++)
                if (idle.t[i] < PSet<uint8_t>::DUMMY) ids[n++] = idle.t[i];
        }
        SSB_CHK(n > 0);
        int j = pool_job(src), s = pool_stage(src);
        SSB_CHK(j >= 0);
        bool sat = jb[j].sat_count == jb[j].n_stages;  // job.saturated, job.py:54-55
        if (s < 0 && !sat) return;
        int dst = sat ? POOL_COMMON : pool_of_job(j);
        for (int i = 0; i < n; i++) {
            move_executor_to_pool(ids[i], dst, false);
            if (dst == POOL_COMMON) {
                detach_executor(j, ids[i]);
                if (p.hist_cap > 0) add_history(ids[i], -1);  // :782
            }
        }
    }
    // _move_executor_to_stage (:799-819) with _try_backup_schedule (:784-797) unrolled into a loop
    __device__ SSB_COLD void move_executor_to_stage(int e, int j, int s)
    {
        for (int guard = 0; guard < 4; guard++) {
            StageRec &r = st[jb[j].node_base + s];
            if (r.remaining == 0) {
                int me = ex[e].job_id, bj, bs;
                SSB_CHK(me != -1);  // _find_backup_stage :823
                if (first_schedulable(true, me, me, bj, bs) || first_schedulable(false, me, me, bj, bs)) {
                    j = bj; s = bs;
                    continue;
                }
                move_idle_executors(ex[e].loc, e);
                return;
            }
            if (ex[e].job_id != j) { send_executor(e, j, s); return; }
            if (!(jb[j].frontier & bit64(s))) {
                ex[e].has_task = 0;
                move_executor_to_pool(e, pool_of_job(j), false);
                return;
            }
            move_executor_to_pool(e, pool_of_stage(j, s), false);
            execute_next_task(e, j, s);
            return;
        }
        fail(1000 + __LINE__);
    }
    __device__ void fulfill_commitment(int e, int dst)  // :699-712
    {
        int src = remove_commitment(e, dst);
        if (h->error) return;
        if (dst == POOL_COMMON) { move_idle_executors(src, e); return; }
        SSB_CHK(dst >= 2 + p.Jc);
        move_executor_to_stage(e, pool_job(dst), pool_stage(dst));
    }
    __device__ void commit_remaining_executors()  // :487-503
    {
        int n = num_committable();
        SSB_CHK(n >= 0);
        if (n > 0) add_commitment(n, POOL_COMMON);
    }
    __device__ void fulfill_commitments_from_source()  // :730-743
    {
        int src = h->source;
        SSB_CHK(src != POOL_NONE);
        PSet<uint8_t> idle = idle_executors(src);
        // snapshot of the source's commitments in insertion order (get_source_commitments(): dict.copy())
        int16_t sn[136];
        int32_t sd[136];
        int ns = 0;
        for (int i = 0; i < h->n_commits && ns < 136; i++)
            if (cm[i].src == src) { sd[ns] = cm[i].dst; sn[ns] = (int16_t)cm[i].n; ns++; }
        for (int k = 0; k < ns; k++) {
            int want = sn[k];
            SSB_CHK(want > 0);
            while (want > 0 && idle.used > 0) {
                int e = ps_pop(idle);
                fulfill_commitment(e, sd[k]);
                if (h->error) return;
                want--;
            }
        }
        SSB_CHK(idle.used == 0);
    }

    // ------------------------------------------------------------ event handlers
    __device__ void handle_job_arrival(int j)  // :428-438 (pools were initialised at reset)
    {
        act[h->n_active++] = (int16_t)j;
        jb[j].state = JOB_ACTIVE;
        if (pool_size(POOL_COMMON) > 0) h->source = POOL_COMMON;
    }
    __device__ void handle_executor_arrival(int e, int j, int s)  // :440-450
    {
        SSB_CHK(!ex[e].has_task);  // job.py:82
        jb[j].n_local += 1;
        ex[e].job_id = (int16_t)j;
        if (p.hist_cap > 0) add_history(e, j);  // :445
        StageRec &r = st[jb[j].node_base + s];
        SSB_CHK(r.moving_to > 0);
        r.moving_to -= 1;  // record_executor_arrival
        update_sat(j, s);
        move_executor_to_pool(e, pool_of_job(j), false);
        move_executor_to_stage(e, j, s);
    }
    __device__ bool record_stage_completion(int j, int s)  // job.py:65-73, :113-128
    {
        JobRec &J = jb[j];
        J.active &= ~bit64(s);
        SSB_CHKR(J.frontier & bit64(s), false);
        J.frontier &= ~bit64(s);
        uint64_t kids = p.b_child[J.ts_base + s] & J.active, fresh = 0;
        const uint64_t *pm = p.b_parent + J.ts_base;
        while (kids) {
            int c = ffs64(kids);
            kids &= kids - 1;
            if ((pm[c] & J.active) == 0) fresh |= bit64(c);  // all parents completed
        }
        J.frontier |= fresh;
        return fresh != 0;
    }
    __device__ void process_job_completion(int j)  // :682-697
    {
        if (pool_size(pool_of_job(j)) > 0) move_idle_executors(pool_of_job(j), -1);
        SSB_CHK(pool_size(pool_of_job(j)) == 0);
        int n = h->n_active, idx = -1;
        for (int i = 0; i < n; i++) if (act[i] == j) { idx = i; break; }
        SSB_CHK(idx >= 0);
        for (int i = idx; i + 1 < n; i++) act[i] = act[i + 1];
        h->n_active = n - 1;
        h->n_completed += 1;
        jb[j].state = JOB_COMPLETED;
        jb[j].sched = 0;
        jb[j].t_completed = h->wall_time;
    }
    __device__ void handle_task_completion(int e, int j, int s)  // :452-483
    {
        StageRec &r = st[jb[j].node_base + s];
        SSB_CHK(r.completed < r.num_tasks);
        r.completed += 1;
        ex[e].is_executing = 0;
        if (r.remaining > 0) { execute_next_task(e, j, s); return; }
        bool frontier_changed = false;
        if (r.completed == r.num_tasks) frontier_changed = record_stage_completion(j, s);
        if (jb[j].active == 0) process_job_completion(j);
        if (h->error) return;
        // _handle_released_executor (:639-660)
        bool had = false;
        int dst = peek_commitment(pool_of_stage(j, s));
        if (dst != POOL_NONE) { fulfill_commitment(e, dst); had = true; }
        else {
            ex[e].has_task = 0;
            if (frontier_changed) move_idle_executors(pool_of_stage(j, s), e);
        }
        // _update_executor_source (:662-674)
        if (frontier_changed) h->source = pool_of_job(j);
        else if (!had) h->source = pool_of_stage(j, s);
    }
    __device__ void log_event(int type, int j, int s, int task, int e, double tacc)
    {
        if (p.log_cap > 0 && h->log_n < p.log_cap) {
            LogRow r;
            r.t = h->wall_time; r.t_acc = tacc; r.task = task; r.job = (int16_t)j; r.stage = (int16_t)s;
            r.exec = (int16_t)e; r.type = (uint8_t)type; r.pad = 0; r.pad1 = 0;
            p.log[(size_t)b * p.log_cap + h->log_n] = r;
        }
        h->log_n += 1;
    }
    // handles popped event `idx` (executor id, or E for the next job arrival) at time t
    __device__ void handle_event(int idx, double t)  // :317-318, :327-329
    {
        h->wall_time = t;
        stats->events++;
        if (idx == p.E) {
            int j = h->next_arrival++;
            log_event(EV_JOB_ARRIVAL, j, -1, -1, -1, __longlong_as_double(0x7ff0000000000000ll));
            handle_job_arrival(j);
            return;
        }
        ExecRec &x = ex[idx];
        int kind = x.ev_kind, j = x.ev_job, s = x.ev_stage;
        x.ev_kind = 0;
        if (kind == EV_TASK_FINISHED) {
            log_event(kind, j, s, x.ev_task, idx, x.t_acc);
            handle_task_completion(idx, j, s);
        } else {
            log_event(kind, j, s, -1, idx, __longlong_as_double(0x7ff0000000000000ll));
            handle_executor_arrival(idx, j, s);
        }
    }

    // ------------------------------------------------------------ timeline: next event by (t, seq)
    __device__ int pop_min_w(double &t_out)
    {
        unsigned long long kt = 0x7ff8000000000000ull;  // > every finite time and +inf
        uint32_t ks = 0xffffffffu;
        int idx = -1;
        for (int e = lane; e < p.E; e += 32) {
            const ExecRec &x = ex[e];
            if (x.ev_kind) {
                unsigned long long t = (unsigned long long)__double_as_longlong(x.ev_t);
                if (t < kt || (t == kt && x.ev_seq < ks)) { kt = t; ks = x.ev_seq; idx = e; }
            }
        }
        if (lane == 31) {  // arrival cursor: arrivals were "pushed" first, seq = job id (:152-154)
            int na = h->next_arrival;
            if (na < h->n_jobs) {
                unsigned long long t = (unsigned long long)__double_as_longlong(jb[na].t_arrival);
                if (t < kt || (t == kt && (uint32_t)na < ks)) { kt = t; ks = (uint32_t)na; idx = p.E; }
            }
        }
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            unsigned long long ot = __shfl_xor_sync(FULL, kt, off);
            uint32_t os = __shfl_xor_sync(FULL, ks, off);
            int oi = __shfl_xor_sync(FULL, idx, off);
            if (ot < kt || (ot == kt && os < ks)) { kt = ot; ks = os; idx = oi; }
        }
        t_out = __longlong_as_double((long long)kt);
        return idx;
    }

    // ------------------------------------------------------------ batched fast path (E <= 32)
    // ~99 % of the timeline events are "executor finishes a task and takes the next task of the same
    // stage" (:464-467).  Such events only touch their own executor and their stage's counters, so a
    // prefix (in (t, seq) order) of the pending events that are all of this kind, that leave their
    // stage's saturation unchanged, and that precede every event the batch itself creates (and the
    // next job arrival) can be handled in ONE warp iteration, one event per lane:
    //   less_e      = bitmask of lanes whose pending event is ordered before lane e's   (all-pairs)
    //   rank_e      = popc(less_e)            launch idx = launch_idx + rank_e (Philox counter / tape)
    //   remaining_e = stage.remaining - popc(less_e & lanes on the same stage)
    //   G           = min over all eligible lanes of their NEW event time
    //   member_e    = eligible, t_e <= G, and no ineligible / later-than-G lane ordered before e
    // The result is identical to handling the events one by one (a shorter prefix is always valid).
    // Measured on C2: 3.8 events per iteration.  Between general-path events everything the loop
    // needs lives in registers, one executor per lane: the pending event, the stage's counters and
    // the two rest-wave duration-table rows the executor-level draw can select; per iteration a lane
    // issues one global load (the sampled duration) and its stores.
    struct HotLane {
        unsigned long long kt;  // event time (f64 bits) and push counter
        double t_acc;
        uint32_t ks;
        int kind, j, s, node, task;
        int rem, comp, mc;   // stage: remaining, completed, moving_to + commit_to
        uint2 oc_a, oc_b;    // rest-wave (offset, count) for the left / right executor level
        int thr, range;      // _sample_executor_key: key = left iff 1 + int(u * range) <= thr
        bool fast_ok;        // this executor's next launch can be sampled without the fallback chain
        bool touched;        // handled at least one event in this fast phase (its t_acc is then that event's time)
        unsigned same;       // lanes whose pending event belongs to the same stage (constant during a fast phase)
        unsigned less;       // lanes whose 32-bit order key is smaller than this lane's (maintained by fast_batch_w)
        uint32_t rx, ry;     // task-stream draws (Philox words x, y) of launch number H.rng_base + lane
    };
    struct HotEnv {  // uniform per-environment scalars
        unsigned long long t_arr;
        double wall;
        long long log_n;
        uint32_t launch_idx, seq;
        int events;
        bool quiet;  // no committable executors at the current (possibly stale) source
        uint32_t rng_base;  // launch number whose draws lane 0 caches (one-slot fast path)
    };
    // (must inline: a non-inlined callee taking L/H by reference would pin them in local memory)
    // slot of executor e (e >= E: an empty slot whose pseudo node id is unique)
    __device__ __forceinline__ void hot_load_slot(HotLane &L, int e)
    {
        L.kt = 0x7ff8000000000000ull; L.ks = 0xffffffffu; L.kind = 0; L.j = 0; L.s = 0;
        L.node = -1 - e; L.task = -1; L.t_acc = 0.0; L.rem = L.comp = L.mc = 0;
        L.oc_a = L.oc_b = make_uint2(0u, 0u); L.thr = L.range = 0; L.fast_ok = false;
        L.touched = false; L.same = 0; L.less = 0;
        if (e < p.E) {
            const ExecRec &x = ex[e];
            L.kind = x.ev_kind;
            if (L.kind) {
                L.kt = (unsigned long long)__double_as_longlong(x.ev_t);
                L.ks = x.ev_seq; L.j = x.ev_job; L.s = x.ev_stage; L.task = x.ev_task; L.t_acc = x.t_acc;
                const JobRec &J = jb[L.j];
                L.node = J.node_base + L.s;
                const StageRec r = st[L.node];
                L.rem = r.remaining; L.comp = r.completed; L.mc = (int)r.moving_to + (int)r.commit_to;
                if (L.kind == EV_TASK_FINISHED) {
                    const int ts = J.ts_base + L.s, n_local = J.n_local;
                    if (h->use_tape) L.fast_ok = true;
                    else if (n_local > 0 && n_local <= p.E) {
                        const short4 iv = p.iv[n_local];
                        const int fw = p.b_present[ts * 4 + 1], rw = p.b_present[ts * 4 + 2];
                        const int top = fw ? 31 - __clz(fw) : -1;  // max(data["first_wave"])
                        int la = iv.z, lb = iv.w;
                        if (la < 0 || !((fw >> la) & 1)) la = top;
                        if (lb < 0 || !((fw >> lb) & 1)) lb = top;
                        if (la >= 0 && ((rw >> la) & 1)) L.oc_a = p.b_dur[(ts * 3 + 2) * 8 + la];
                        if (lb >= 0 && ((rw >> lb) & 1)) L.oc_b = p.b_dur[(ts * 3 + 2) * 8 + lb];
                        L.range = iv.y - iv.x;
                        L.thr = n_local - iv.x;
                        // the rest-wave list must exist for every level the draw can pick
                        L.fast_ok = L.oc_a.y > 0 && (L.range == 0 || L.oc_b.y > 0);
                    }
                }
            }
        }
    }
    __device__ __forceinline__ void hot_load_env(HotEnv &H)
    {
        H.t_arr = 0x7ff0000000000000ull;
        int na = h->next_arrival;
        if (na < h->n_jobs) H.t_arr = (unsigned long long)__double_as_longlong(jb[na].t_arrival);
        H.wall = h->wall_time; H.log_n = h->log_n; H.launch_idx = h->launch_idx; H.seq = h->seq;
        H.events = 0;
        H.quiet = num_committable() == 0;
    }
    // The task stream is counter-based, so the draws of the next 32 launches can be produced by the 32 lanes at
    // once and handed out by shuffle: one Philox evaluation per 32 launches instead of one per loop iteration.
    __device__ __forceinline__ void hot_refill_rng(HotLane &L, HotEnv &H)
    {
        H.rng_base = H.launch_idx;
        const uint4 w = philox4x32_10(H.rng_base + (uint32_t)lane, 0u, 2u, 0u, (uint32_t)h->seed, (uint32_t)(h->seed >> 32));
        L.rx = w.x; L.ry = w.y;
    }
    // order of the pending events by (t, push counter) (event.py:34-35): a 32-bit fixed-point key, floor(16 t)
    // saturated, almost always decides (event times are mostly whole milliseconds, which tie in the upper f64 word
    // above 2^20 ms); equal keys take the exact path.  Empty slots sort last.
    __device__ __forceinline__ uint32_t order_key(const HotLane &L) const
    {
        return L.kind ? __double2uint_rd(__dmul_rn(__longlong_as_double((long long)L.kt), 16.0)) : 0xffffffffu;
    }
    __device__ __forceinline__ void hot_load(HotLane &L, HotEnv &H)
    {
        hot_load_slot(L, lane);
        hot_load_env(H);
        L.same = __match_any_sync(FULL, L.node);
        if (H.quiet) {
            // all-pairs order masks on the 32-bit keys, ONCE per fast phase; fast_batch_w maintains them
            // (kept rolled on purpose: instruction fetch, not shuffle latency, bounds this code -- the
            // unrolled form measured 6475 vs 4266 cycles per iteration, profiles/r01_ab_unroll.txt)
            const uint32_t hi = order_key(L);
            unsigned less = 0;
#pragma unroll 1
            for (int i = 0; i < p.E; i++) less |= (__shfl_sync(FULL, hi, i) < hi) ? (1u << i) : 0u;
            L.less = less;
        }
        L.rx = L.ry = 0u; H.rng_base = H.launch_idx;
        if (H.quiet && !h->use_tape) hot_refill_rng(L, H);
    }
    // one-slot fast phase: the wall time is the time of the last event handled, i.e. the maximum over the
    // lanes that handled one of their t_acc (non-negative doubles order like their bit patterns)
    __device__ __forceinline__ void hot_flush1(const HotLane &L, HotEnv &H)
    {
        if (H.events) {
            const unsigned long long tb = L.touched ? (unsigned long long)__double_as_longlong(L.t_acc) : 0ull;
            const uint32_t whi = __reduce_max_sync(FULL, (uint32_t)(tb >> 32));
            const uint32_t wlo = __reduce_max_sync(FULL, (uint32_t)(tb >> 32) == whi ? (uint32_t)tb : 0u);
            H.wall = __longlong_as_double((long long)(((unsigned long long)whi << 32) | wlo));
        }
        hot_flush(H);
    }
    __device__ __forceinline__ void hot_flush(const HotEnv &H)
    {
        if (lane == 0 && H.events) {
            h->wall_time = H.wall; h->log_n = H.log_n; h->launch_idx = H.launch_idx; h->seq = H.seq;
            stats->events += (unsigned long long)H.events;
        }
        __syncwarp();
    }
    // exact (t, seq) order, used when two pending events agree in the upper half of their timestamps
    __device__ SSB_RARE unsigned exact_less_w(unsigned long long kt, uint32_t ks)
    {
        unsigned less = 0;
        for (int i = 0; i < p.E; i++) {
            unsigned long long ot = __shfl_sync(FULL, kt, i);
            uint32_t os = __shfl_sync(FULL, ks, i);
            less |= (unsigned)(ot < kt || (ot == kt && os < ks)) << i;
        }
        return less;
    }
    __device__ SSB_RARE void log_batch_row(long long row, double t, double t_acc, int task, int j, int s, int e)
    {
        if (row >= p.log_cap) return;
        LogRow r;
        r.t = t; r.t_acc = t_acc; r.task = task; r.job = (int16_t)j; r.stage = (int16_t)s;
        r.exec = (int16_t)e; r.type = (uint8_t)EV_TASK_FINISHED; r.pad = 0; r.pad1 = 0;
        p.log[(size_t)b * p.log_cap + row] = r;
    }
    __device__ __forceinline__ int fast_batch_w(HotLane &L, HotEnv &H, int budget)
    {
        const unsigned long long INF_BITS = 0x7ff0000000000000ull;
        if (!H.quiet) return 0;
        const bool pending = L.kind != 0;
        const unsigned pend_mask = __ballot_sync(FULL, pending);
        if (!pend_mask) return 0;
        // order masks: maintained across iterations on the 32-bit keys (hot_load computes them once per phase, the
        // end of this function updates them for the members); the full all-pairs loop per iteration was 21 % of all
        // instructions the rollout kernel executed (profiles/r02_ncu_rollout_v5_by_line.txt).  Equal keys among the
        // pending events: exact (t, seq) order for this iteration.
        const uint32_t hi = order_key(L);
        unsigned less = L.less;
        {
            const unsigned eq = __match_any_sync(FULL, hi) & pend_mask;
            if (__any_sync(FULL, pending && (eq & (eq - 1)))) less = exact_less_w(L.kt, L.ks);
        }
        less &= pend_mask;
        const int rank = __popc(less);
        const unsigned same_node = L.same;
        const int before_same = __popc(less & same_node);
        // eligibility: TASK_FINISHED before the next arrival (an arrival at the same time pops first,
        // its seq is smaller), tasks left after this launch, saturation bit of the stage unchanged
        const int rem = L.rem - before_same;
        bool elig = pending && L.fast_ok && L.kt < H.t_arr && rank < budget && rem > 1 &&
                    ((rem <= L.mc) == (rem - 1 <= L.mc));
        const double t = __longlong_as_double((long long)L.kt);
        double d = 0.0;
        unsigned long long nt = INF_BITS;
        const bool tape = h->use_tape;
        const uint32_t li = H.launch_idx + (uint32_t)rank;
        uint32_t wx = 0u, wy = 0u;
        if (!tape) {  // draws of launch li: cached by lane li - rng_base (refilled when the window runs out)
            if (H.launch_idx + (uint32_t)__popc(pend_mask) > H.rng_base + 32u) hot_refill_rng(L, H);
            const int src = (int)(li - H.rng_base) & 31;
            wx = __shfl_sync(FULL, L.rx, src);
            wy = __shfl_sync(FULL, L.ry, src);
        }
        if (elig) {
            if (tape) {
                if ((int)li < h->tape_len) d = p.tape[(size_t)b * p.tape_cap + li];
                else elig = false;  // the general path reports the exhausted tape
            } else {  // tpch.py:75-106 for an executor continuing on its stage: rest_wave[level]
                uint2 oc = L.oc_a;
                if (L.range) {
                    double u = __dmul_rn((double)wx, 1.0 / 4294967296.0);
                    int rand_pt = 1 + (int)__dmul_rn(u, (double)L.range);
                    if (rand_pt > L.thr) oc = L.oc_b;
                }
                d = p.b_vals[oc.x + bounded(wy, oc.y)];
            }
            if (elig) nt = (unsigned long long)__double_as_longlong(__dadd_rn(t, d));
        }
        // G = earliest event the batch could create (non-negative doubles order like their bit patterns)
        const uint32_t ghi = __reduce_min_sync(FULL, (uint32_t)(nt >> 32));
        const uint32_t glo = __reduce_min_sync(FULL, (uint32_t)(nt >> 32) == ghi ? (uint32_t)nt : 0xffffffffu);
        const unsigned long long G = ((unsigned long long)ghi << 32) | glo;
        const unsigned bad = __ballot_sync(FULL, pending && (!elig || L.kt > G));
        const bool member = pending && !((bad >> lane) & 1) && !(less & bad);
        const unsigned mem_mask = __ballot_sync(FULL, member);
        const int m = __popc(mem_mask);
        if (m == 0) return 0;
        const int cnt = __popc(same_node & mem_mask);  // launches of my stage in this batch
        if (member) {
            if (p.log_cap > 0) log_batch_row(H.log_n + rank, t, L.t_acc, L.task, L.j, L.s, lane);
            L.kt = nt; L.t_acc = t; L.ks = H.seq + (uint32_t)rank; L.task = rem - 1; L.touched = true;
            ExecRec &x = ex[lane];
            x.ev_t = __longlong_as_double((long long)nt); x.t_acc = t; x.ev_seq = L.ks; x.ev_task = L.task;
            if (before_same == cnt - 1) {  // last launch of this stage in the batch: it owns the counters
                StageRec &r = st[L.node];
                r.remaining = (uint16_t)(L.rem - cnt);
                r.completed = (uint16_t)(L.comp + cnt);
                r.mrd = (float)d;
            }
        }
        L.rem -= cnt; L.comp += cnt;  // every lane on that stage tracks its counters
        // (the wall time -- the time of the last member -- is taken once per phase, in hot_flush1)
        H.launch_idx += (uint32_t)m; H.seq += (uint32_t)m; H.log_n += m; H.events += m;
        {
            // key masks for the next iteration: only the members' keys changed.  For member u: bit u of every
            // lane's mask = "u's new key is smaller than mine"; u's own mask = the lanes whose key it does not exceed
            // ... complemented: the lanes with a smaller key (equal keys: neither side, as in the full loop).
            L.kt = member ? nt : L.kt;  // (already assigned above for members; keeps the compiler's view simple)
            const uint32_t hi2 = order_key(L);
            unsigned nl = L.less, mm = mem_mask;
#pragma unroll 1
            while (mm) {
                const int u = __ffs((int)mm) - 1;
                mm &= mm - 1;
                const uint32_t ku = __shfl_sync(FULL, hi2, u);
                const unsigned smaller = __ballot_sync(FULL, hi2 < ku);  // lanes whose key is smaller than u's
                nl = ku < hi2 ? (nl | (1u << u)) : (nl & ~(1u << u));
                if (lane == u) nl = smaller;
            }
            L.less = nl;
        }
        return m;
    }


    // ------------------------------------------------------------ batched fast path, 32 < E <= 64
    // Same algorithm with two executors per lane: slot A = executor `lane`, slot B = executor
    // `lane + 32`.  Order masks come in four flavours xy = "lanes whose slot-y event precedes my slot-x
    // event".  The stage of a slot does not change during a fast phase, so the same-stage masks are
    // built once per phase.
    struct Same2 { unsigned aa, ab, ba, bb; };
    __device__ __forceinline__ void same_nodes2_w(const HotLane &A, const HotLane &Bq, Same2 &S)
    {
        S.aa = S.ab = S.ba = S.bb = 0;
#pragma unroll 1
        for (int i = 0; i < 32; i++) {
            const int na = __shfl_sync(FULL, A.node, i), nb = __shfl_sync(FULL, Bq.node, i);
            const unsigned bit = 1u << i;
            S.aa |= na == A.node ? bit : 0u;  S.ab |= nb == A.node ? bit : 0u;
            S.ba |= na == Bq.node ? bit : 0u; S.bb |= nb == Bq.node ? bit : 0u;
        }
    }
    // exact (t, seq) order masks, used when two pending events agree in the upper timestamp word
    __device__ SSB_RARE void exact_less2_w(unsigned long long kta, uint32_t ksa, unsigned long long ktb,
                                            uint32_t ksb, unsigned *out)
    {
        unsigned aa = 0, ab = 0, ba = 0, bb = 0;
        for (int i = 0; i < 32; i++) {
            const unsigned long long ota = __shfl_sync(FULL, kta, i), otb = __shfl_sync(FULL, ktb, i);
            const uint32_t osa = __shfl_sync(FULL, ksa, i), osb = __shfl_sync(FULL, ksb, i);
            const unsigned bit = 1u << i;
            aa |= (ota < kta || (ota == kta && osa < ksa)) ? bit : 0u;
            ab |= (otb < kta || (otb == kta && osb < ksa)) ? bit : 0u;
            ba |= (ota < ktb || (ota == ktb && osa < ksb)) ? bit : 0u;
            bb |= (otb < ktb || (otb == ktb && osb < ksb)) ? bit : 0u;
        }
        out[0] = aa; out[1] = ab; out[2] = ba; out[3] = bb;
    }
    // The 32-bit order keys tie (with 50 pending events equal event times are common): instead of redoing all 64 x 64
    // comparisons exactly (exact_less2_w), find the lanes that hold a pending event whose key equals one of another
    // pending event's keys (U) and redo the comparisons against THOSE lanes only, on the full (t, seq) pairs.  Pairs
    // whose keys differ are ordered by the keys (floor(16 t) is monotone in t), so the masks come out exact.
    __device__ SSB_RARE void refine_ties2_w(uint32_t hia, uint32_t hib, bool pa, bool pb, unsigned penda, unsigned pendb,
                                             unsigned long long kta, uint32_t ksa, unsigned long long ktb, uint32_t ksb,
                                             unsigned *m)
    {
        unsigned tie = 0;
#pragma unroll 1
        for (int i = 0; i < 32; i++) {
            const uint32_t oa = __shfl_sync(FULL, hia, i), ob = __shfl_sync(FULL, hib, i);
            const bool ia = (penda >> i) & 1, ib = (pendb >> i) & 1;
            const bool t = (pa && ((ia && oa == hia && i != lane) || (ib && ob == hia))) ||
                           (pb && ((ia && oa == hib) || (ib && ob == hib && i != lane)));
            tie |= t ? 1u << i : 0u;
        }
        unsigned U = __reduce_or_sync(FULL, tie);
        unsigned aa = m[0], ab = m[1], ba = m[2], bb = m[3];
        while (U) {
            const int i = __ffs((int)U) - 1;
            U &= U - 1;
            const unsigned long long ota = __shfl_sync(FULL, kta, i), otb = __shfl_sync(FULL, ktb, i);
            const uint32_t osa = __shfl_sync(FULL, ksa, i), osb = __shfl_sync(FULL, ksb, i);
            const unsigned bit = 1u << i;
            aa = (aa & ~bit) | ((ota < kta || (ota == kta && osa < ksa)) ? bit : 0u);
            ab = (ab & ~bit) | ((otb < kta || (otb == kta && osb < ksa)) ? bit : 0u);
            ba = (ba & ~bit) | ((ota < ktb || (ota == ktb && osa < ksb)) ? bit : 0u);
            bb = (bb & ~bit) | ((otb < ktb || (otb == ktb && osb < ksb)) ? bit : 0u);
        }
        m[0] = aa; m[1] = ab; m[2] = ba; m[3] = bb;
    }
    __device__ __forceinline__ int fast_batch2_w(HotLane &A, HotLane &Bq, const Same2 &S, HotEnv &H, int budget)
    {
        const unsigned long long INF_BITS = 0x7ff0000000000000ull;
        if (!H.quiet) return 0;
        const bool pa = A.kind != 0, pb = Bq.kind != 0;
        const unsigned penda = __ballot_sync(FULL, pa), pendb = __ballot_sync(FULL, pb);
        if (!(penda | pendb)) return 0;
        // 32-bit fixed-point order keys floor(16 t), saturated (see fast_batch_w); empty slots sort last
        const uint32_t hia = pa ? __double2uint_rd(__dmul_rn(__longlong_as_double((long long)A.kt), 16.0)) : 0xffffffffu;
        const uint32_t hib = pb ? __double2uint_rd(__dmul_rn(__longlong_as_double((long long)Bq.kt), 16.0)) : 0xffffffffu;
        unsigned aa = 0, ab = 0, ba = 0, bb = 0;
#pragma unroll 1
        for (int i = 0; i < 32; i++) {
            const uint32_t oa = __shfl_sync(FULL, hia, i), ob = __shfl_sync(FULL, hib, i);
            const unsigned bit = 1u << i;
            aa |= oa < hia ? bit : 0u; ab |= ob < hia ? bit : 0u;
            ba |= oa < hib ? bit : 0u; bb |= ob < hib ? bit : 0u;
        }
        aa &= penda; ab &= pendb; ba &= penda; bb &= pendb;
        int ranka = __popc(aa) + __popc(ab), rankb = __popc(ba) + __popc(bb);
        {
            // events that agree in the upper word get equal ranks, so the ranks of the pending events
            // are a permutation of 0..n-1 exactly when the upper words decided every comparison
            const int n = __popc(penda) + __popc(pendb);
            const unsigned long long mine = (pa ? 1ull << ranka : 0ull) | (pb ? 1ull << rankb : 0ull);
            const unsigned long long seen = (unsigned long long)__reduce_or_sync(FULL, (uint32_t)mine) |
                                            ((unsigned long long)__reduce_or_sync(FULL, (uint32_t)(mine >> 32)) << 32);
            if (seen != (n >= 64 ? ~0ull : (1ull << n) - 1ull)) {
                unsigned ex4[4] = {aa, ab, ba, bb};
                refine_ties2_w(hia, hib, pa, pb, penda, pendb, A.kt, A.ks, Bq.kt, Bq.ks, ex4);
                aa = ex4[0] & penda; ab = ex4[1] & pendb; ba = ex4[2] & penda; bb = ex4[3] & pendb;
                ranka = __popc(aa) + __popc(ab); rankb = __popc(ba) + __popc(bb);
            }
        }
        const int bsa = __popc(aa & S.aa) + __popc(ab & S.ab), bsb = __popc(ba & S.ba) + __popc(bb & S.bb);
        const int rema = A.rem - bsa, remb = Bq.rem - bsb;
        bool ea = pa && A.fast_ok && A.kt < H.t_arr && ranka < budget && rema > 1 &&
                  ((rema <= A.mc) == (rema - 1 <= A.mc));
        bool eb = pb && Bq.fast_ok && Bq.kt < H.t_arr && rankb < budget && remb > 1 &&
                  ((remb <= Bq.mc) == (remb - 1 <= Bq.mc));
        const double ta = __longlong_as_double((long long)A.kt), tb = __longlong_as_double((long long)Bq.kt);
        double da = 0.0, db = 0.0;
        // durations of the two slots, one after the other through the same (rolled) code
#pragma unroll 1
        for (int k = 0; k < 2; k++) {
            bool el = k ? eb : ea;
            double d = 0.0;
            if (el) {
                const uint32_t li = H.launch_idx + (uint32_t)(k ? rankb : ranka);
                if (h->use_tape) {
                    if ((int)li < h->tape_len) d = p.tape[(size_t)b * p.tape_cap + li];
                    else el = false;  // the general path reports the exhausted tape
                } else {
                    const uint4 w = philox4x32_10(li, 0u, 2u, 0u, (uint32_t)h->seed, (uint32_t)(h->seed >> 32));
                    uint2 oc = k ? Bq.oc_a : A.oc_a;
                    const int range = k ? Bq.range : A.range;
                    if (range) {
                        double u = __dmul_rn((double)w.x, 1.0 / 4294967296.0);
                        int rand_pt = 1 + (int)__dmul_rn(u, (double)range);
                        if (rand_pt > (k ? Bq.thr : A.thr)) oc = k ? Bq.oc_b : A.oc_b;
                    }
                    d = p.b_vals[oc.x + bounded(w.y, oc.y)];
                }
            }
            if (k) { eb = el; db = d; } else { ea = el; da = d; }
        }
        const unsigned long long nta = ea ? (unsigned long long)__double_as_longlong(__dadd_rn(ta, da)) : INF_BITS;
        const unsigned long long ntb = eb ? (unsigned long long)__double_as_longlong(__dadd_rn(tb, db)) : INF_BITS;
        const unsigned long long ntm = nta < ntb ? nta : ntb;
        const uint32_t ghi = __reduce_min_sync(FULL, (uint32_t)(ntm >> 32));
        const uint32_t glo = __reduce_min_sync(FULL, (uint32_t)(ntm >> 32) == ghi ? (uint32_t)ntm : 0xffffffffu);
        const unsigned long long G = ((unsigned long long)ghi << 32) | glo;
        const unsigned bada = __ballot_sync(FULL, pa && (!ea || A.kt > G));
        const unsigned badb = __ballot_sync(FULL, pb && (!eb || Bq.kt > G));
        const bool ma = pa && !((bada >> lane) & 1) && !(aa & bada) && !(ab & badb);
        const bool mb = pb && !((badb >> lane) & 1) && !(ba & bada) && !(bb & badb);
        const unsigned mema = __ballot_sync(FULL, ma), memb = __ballot_sync(FULL, mb);
        const int m = __popc(mema) + __popc(memb);
        if (m == 0) return 0;
        const int cnta = __popc(S.aa & mema) + __popc(S.ab & memb);
        const int cntb = __popc(S.ba & mema) + __popc(S.bb & memb);
        if (ma) {
            if (p.log_cap > 0) log_batch_row(H.log_n + ranka, ta, A.t_acc, A.task, A.j, A.s, lane);
            A.kt = nta; A.t_acc = ta; A.ks = H.seq + (uint32_t)ranka; A.task = rema - 1;
            ExecRec &x = ex[lane];
            x.ev_t = __longlong_as_double((long long)nta); x.t_acc = ta; x.ev_seq = A.ks; x.ev_task = A.task;
            if (bsa == cnta - 1) {  // last launch of this stage in the batch: it owns the counters
                StageRec &r = st[A.node];
                r.remaining = (uint16_t)(A.rem - cnta);
                r.completed = (uint16_t)(A.comp + cnta);
                r.mrd = (float)da;
            }
        }
        if (mb) {
            if (p.log_cap > 0) log_batch_row(H.log_n + rankb, tb, Bq.t_acc, Bq.task, Bq.j, Bq.s, lane + 32);
            Bq.kt = ntb; Bq.t_acc = tb; Bq.ks = H.seq + (uint32_t)rankb; Bq.task = remb - 1;
            ExecRec &x = ex[lane + 32];
            x.ev_t = __longlong_as_double((long long)ntb); x.t_acc = tb; x.ev_seq = Bq.ks; x.ev_task = Bq.task;
            if (bsb == cntb - 1) {
                StageRec &r = st[Bq.node];
                r.remaining = (uint16_t)(Bq.rem - cntb);
                r.completed = (uint16_t)(Bq.comp + cntb);
                r.mrd = (float)db;
            }
        }
        A.rem -= cnta; A.comp += cnta; Bq.rem -= cntb; Bq.comp += cntb;
        // wall time = time of the last member (non-negative doubles order like their bit patterns)
        const unsigned long long tma = ma ? (unsigned long long)__double_as_longlong(ta) : 0ull;
        const unsigned long long tmb = mb ? (unsigned long long)__double_as_longlong(tb) : 0ull;
        const unsigned long long tmx = tma > tmb ? tma : tmb;
        const uint32_t whi = __reduce_max_sync(FULL, (uint32_t)(tmx >> 32));
        const uint32_t wlo = __reduce_max_sync(FULL, (uint32_t)(tmx >> 32) == whi ? (uint32_t)tmx : 0u);
        H.wall = __longlong_as_double((long long)(((unsigned long long)whi << 32) | wlo));
        H.launch_idx += (uint32_t)m; H.seq += (uint32_t)m; H.log_n += m; H.events += m;
        return m;
    }
    // one fast phase with two slots per lane; returns the number of events it handled
    __device__ __forceinline__ int fast_phase2_w(int budget)
    {
        HotEnv H;
        hot_load_env(H);
        if (!H.quiet) return 0;
        HotLane A, Bq;
        Same2 S;
        hot_load_slot(A, lane);
        hot_load_slot(Bq, lane + 32);
        same_nodes2_w(A, Bq, S);
        int used = 0;
        for (;;) {
            const int m = fast_batch2_w(A, Bq, S, H, budget - used);
            used += m;
            if (m == 0 || used == budget) break;
        }
        hot_flush(H);
        return used;
    }

    // ------------------------------------------------------------ _resume_simulation (:320-343)
    // Returns false when `max_events` (> 0) events were processed without reaching the next
    // scheduling decision: the environment is then "pending" and a later call continues here.
    // NS = executor slots per lane of the batched fast path: 1 serves E <= 32, 2 serves E <= 64
    // (separate kernel instantiations, so that the one-slot kernels keep their register budget).
    template <int NS>
    __device__ bool resume_simulation_w(int max_events)
    {
        int budget = max_events > 0 ? max_events : 0x7fffffff;
        const bool use_fast = NS == 1 ? p.E <= 32 : p.E <= 64;
        for (;;) {
            if constexpr (NS == 2) {
                if (use_fast && budget > 0) budget -= fast_phase2_w(budget);
            } else if (use_fast && budget > 0) {
                // registers only: L and H die before the general path below is entered
                HotLane L;
                HotEnv H;
                SSB_T0();
                hot_load(L, H);
                SSB_TACC(11);
                for (;;) {
                    int m = fast_batch_w(L, H, budget);
                    budget -= m;
                    SSB_TCNT(1, 1);
                    if (m == 0 || budget == 0) break;
                }
                hot_flush1(L, H);
                SSB_TACC(0);
            }
            SSB_T0();
            double t;
            int idx = pop_min_w(t);
            if (idx < 0) break;
            if (budget-- == 0) return false;
            if (lane == 0) handle_event(idx, t);
            __syncwarp();
            SSB_TACC(2);
            SSB_TCNT(3, 1);
            if (h->error) break;
            if (num_committable() <= 0) continue;
            int n = find_schedulable_all_w();
            if (n) { SSB_TACC(4); break; }
            if (lane == 0) { move_idle_executors(POOL_NONE, -1); h->source = POOL_NONE; }
            __syncwarp();
            SSB_TACC(4);
            if (h->error) break;
        }
        return true;
    }

    // ------------------------------------------------------------ reward (:847-874)
    // continuously discounted job-time of one job over [a, b] after the step's start (:866-869)
    __device__ SSB_RARE double discounted_term(double a, double b) const
    {
        return exp(-p.beta * 1e-3 * a) - exp(-p.beta * 1e-3 * b);
    }
    // Lane 0: writes the job ids of set(active_old + active_new) in CPython's iteration order to
    // `ord` and returns their number (:855-858).  Both lists ascend and jobs that arrived during the
    // step have larger ids than every old one, so the distinct ids are inserted in ascending order; the
    // table sizes go 8 -> 32 -> 128 -> 512 -> ... at 5, 19, 77, 307, ... elements, and once every id is
    // smaller than the final table size each id sits in its own slot => iteration is ascending
    // (tests/test_pyset.py checks the claims against the interpreter).  Small sets are emulated in
    // registers, anything else with the generic set emulation.
    // (the ascending case is handled by compute_jobtime_w without materialising the order)
    __device__ SSB_COLD int reward_order(int16_t *ord, int n, int max_id)
    {
        const int16_t *old = p.old_act + (size_t)b * p.Jc;
        const int n_old = h->n_old_active, n_new = h->n_active;
        const int last_old = n_old ? old[n_old - 1] : -1;
        int k = 0;
        if (n <= 18 && max_id < 255) {
            // 8- or 32-slot table without deletions, in registers: keys as bytes of u64 words, occupancy
            // as a bit mask, so the 9-slot linear probe of set_add_entry is one find-first-zero
            uint64_t t8 = 0, T0 = 0, T1 = 0, T2 = 0, T3 = 0;
            uint32_t occ8 = 0, occ = 0;
            int cnt = 0;
            bool big = false;
            auto put32 = [&](int key) {
                unsigned perturb = (unsigned)key, i = (unsigned)key & 31u;
                for (;;) {
                    if (!((occ >> i) & 1u)) break;
                    if (i + 9 <= 31) {
                        unsigned m = (~occ >> (i + 1)) & 0x1ffu;
                        if (m) { i = i + (unsigned)__ffs((int)m); break; }
                    }
                    perturb >>= 5;
                    i = (i * 5 + 1 + perturb) & 31u;
                }
                occ |= 1u << i;
                const uint64_t v = (uint64_t)key << (8 * (i & 7));
                const unsigned wsel = i >> 3;
                T0 |= wsel == 0 ? v : 0ull; T1 |= wsel == 1 ? v : 0ull;
                T2 |= wsel == 2 ? v : 0ull; T3 |= wsel == 3 ? v : 0ull;
            };
            auto put = [&](int key) {
                if (big) { put32(key); cnt++; return; }
                unsigned perturb = (unsigned)key, i = (unsigned)key & 7u;  // mask 7: no linear probes
                while ((occ8 >> i) & 1u) { perturb >>= 5; i = (i * 5 + 1 + perturb) & 7u; }
                occ8 |= 1u << i;
                t8 |= (uint64_t)key << (8 * i);
                if (++cnt == 5) {  // fill*5 >= mask*3: resize to 32, re-insert in old slot order
                    for (int s = 0; s < 8; s++)
                        if ((occ8 >> s) & 1u) put32((int)((t8 >> (8 * s)) & 0xff));
                    big = true;
                }
            };
            for (int i = 0; i < n_old; i++) put(old[i]);
            for (int i = 0; i < n_new; i++) if (act[i] > last_old) put(act[i]);
            if (!big) {
                for (int s = 0; s < 8; s++)
                    if ((occ8 >> s) & 1u) ord[k++] = (int16_t)((t8 >> (8 * s)) & 0xff);
            } else {
                for (int s = 0; s < 32; s++) {
                    if (!((occ >> s) & 1u)) continue;
                    const uint64_t wv = (s >> 3) == 0 ? T0 : (s >> 3) == 1 ? T1 : (s >> 3) == 2 ? T2 : T3;
                    ord[k++] = (int16_t)((wv >> (8 * (s & 7))) & 0xff);
                }
            }
            return k;
        }
        uint16_t *tab = p.rset + (size_t)b * 2 * p.RT, *tmp = tab + p.RT;
        PSet<uint16_t> ids;
        ps_init(ids, tab);
#pragma unroll 1
        for (int i = 0; i < n_old; i++) ps_add(ids, old[i], tmp);
        // (the new list = survivors of the old one, already in the set, + the arrivals, whose ids are larger)
#pragma unroll 1
        for (int i = 0; i < n_new; i++) if (act[i] > last_old) ps_add(ids, act[i], tmp);
        for (int i = 0; i <= ids.mask; i++)
            if (ids.t[i] < PSet<uint16_t>::DUMMY) ord[k++] = (int16_t)ids.t[i];
        return k;
    }
    // _compute_jobtime: lane 0 fixes the summation order, all lanes fetch their jobs' overlap with the
    // step in parallel, and the f64 sum is taken sequentially in that order (bit-identical to the loop)
    __device__ double compute_jobtime_w()
    {
        const double wall = h->wall_time, wall_old = h->wall_old;
        if (wall - wall_old == 0.0) return 0.0;
        int16_t *ord = p.reward_ord + (size_t)b * p.Jc;
        // distinct ids = the old list, then the jobs that arrived during the step (the tail of act)
        const int16_t *old = p.old_act + (size_t)b * p.Jc;
        const int n_old = h->n_old_active, n_new = h->n_active;
        const int last_old = n_old ? old[n_old - 1] : -1;
        int n_arr = 0;
        while (n_arr < n_new && act[n_new - 1 - n_arr] > last_old) n_arr++;
        int n = n_old + n_arr;
        const int max_id = n_arr ? act[n_new - 1] : last_old;
        const int F = n < 5 ? 8 : n < 19 ? 32 : n < 77 ? 128 : n < 307 ? 512 : n < 1229 ? 2048 : 0;
        const bool ascending = max_id < F;  // every id in its own slot of the final table
        // Small sets (n < 19: an 8- or 32-slot table) whose ids are distinct modulo the table size also sit each
        // in its own slot, id & mask, whatever the insertion order -> iteration order = slot order
        // (tests/test_pyset.py::test_small_set_slot_order checks this against the interpreter).
        bool by_slot = false;
        int src = lane;  // lane whose term is summed at position `lane`
        if (!ascending && n < 19) {
            const int mask = n < 5 ? 7 : 31;
            const int key = lane < n ? (lane < n_old ? old[lane] : act[n_new - n_arr + (lane - n_old)]) : -1 - lane;
            const int slot = lane < n ? (key & mask) : 32 + lane;
            const unsigned same = __match_any_sync(FULL, slot);
            if (!__any_sync(FULL, same & (same - 1))) {
                by_slot = true;
                const unsigned occ = __ballot_sync(FULL, lane < n) ? __reduce_or_sync(FULL, lane < n ? 1u << slot : 0u) : 0u;
                const int pos = lane < n ? __popc(occ & ((1u << slot) - 1u)) : 32;
                for (int k = 0; k < n; k++)
                    if (__shfl_sync(FULL, pos, k) == lane) src = k;
            }
        }
        if (!ascending && !by_slot) {
            int m = 0;
            if (lane == 0) m = reward_order(ord, n, max_id);
            n = __shfl_sync(FULL, m, 0);
            __syncwarp();
        }
        const double beta = p.beta;
        double jt = 0.0;
        for (int base = 0; base < n; base += 32) {
            double term = 0.0;
            if (base + lane < n) {
                const int k = base + lane;
                const int j = (!ascending && !by_slot) ? ord[k] : k < n_old ? old[k] : act[n_new - n_arr + (k - n_old)];
                const double start = fmax(jb[j].t_arrival, wall_old), end = fmin(jb[j].t_completed, wall);
                term = beta == 0.0 ? __dadd_rn(end, -start) : discounted_term(start - wall_old, end - wall_old);
            }
            if (by_slot) term = __shfl_sync(FULL, term, src);  // n <= 18: a single chunk
            const int m = min(32, n - base);
            for (int i = 0; i < m; i++) jt = __dadd_rn(jt, __shfl_sync(FULL, term, i));
        }
        if (beta > 0.0) jt /= beta;
        return jt;
    }

    // ------------------------------------------------------------ _observe (:345-406, utils.py:5-22)
    // edges of a job's template (ne entries from eb) with both ends active: the job's edges in the observation
    // (utils.subgraph, utils.py:5-22); one thread per job
    __device__ int job_obs_edges(uint64_t active, int eb, int ne) const
    {
        int c = 0;
#pragma unroll 8
        for (int k = 0; k < ne; k++) {
            const int u = p.b_edges[2 * (eb + k)], v = p.b_edges[2 * (eb + k) + 1];
            c += (int)((active >> u) & (active >> v) & 1);
        }
        return c;
    }
    // What observe_w writes: OBS_FULL = header, observation counters and the graph slabs (dag_ptr, exec_supplies,
    // nodes, edge_links).  The fused rollout splits it: OBS_HDR every decision (the header and the counters, from
    // a count pass with one lane per active job), OBS_GRAPH once when its decision loop ends (the slabs only).
    enum : int { OBS_HDR = 1, OBS_GRAPH = 2, OBS_FULL = OBS_HDR | OBS_GRAPH };
    template <int PARTS = OBS_FULL>
    __device__ SSB_COLD void observe_w(double reward, bool terminated)
    {
        const int n_active = h->n_active;
        float *nodes = p.obs_nodes + (size_t)b * p.Sc * 3;
        int32_t *edges = p.obs_edges + (size_t)b * p.Mc * 2;
        int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
        int32_t *sup = p.obs_supplies + (size_t)b * p.Jc;
        const int src_job = source_job_id();
        int src_idx = n_active, N = 0, M = 0;
        if constexpr (PARTS == OBS_HDR) {
            for (int base = 0; base < n_active; base += 32) {
                const int i = base + lane;
                int j = -1;
                if (i < n_active) {
                    j = act[i];
                    const JobRec &J = jb[j];
                    const uint64_t active = J.active;
                    const int eb = p.b_edge_base[J.tmpl];
                    N += popc64(active);
                    M += job_obs_edges(active, eb, p.b_edge_base[J.tmpl + 1] - eb);
                }
                unsigned hit = __ballot_sync(FULL, j >= 0 && j == src_job);
                if (hit) src_idx = base + __ffs(hit) - 1;
            }
            N = __reduce_add_sync(FULL, N);
            M = __reduce_add_sync(FULL, M);
        } else {
            // dag_ptr / exec_supplies / source_job_idx: exclusive scan of per-job active-stage counts
            for (int base = 0; base < n_active; base += 32) {
                int i = base + lane, cnt = 0, j = -1;
                if (i < n_active) {
                    j = act[i];
                    cnt = popc64(jb[j].active);
                    sup[i] = jb[j].supply;
                }
                int incl = cnt;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    int v = __shfl_up_sync(FULL, incl, off);
                    if (lane >= off) incl += v;
                }
                if (i < n_active) dag_ptr[i + 1] = N + incl;
                unsigned hit = __ballot_sync(FULL, j >= 0 && j == src_job);
                if (hit) src_idx = base + __ffs(hit) - 1;
                N += __shfl_sync(FULL, incl, 31);
            }
            if (lane == 0) dag_ptr[0] = 0;
            __syncwarp();
            // nodes and edges, one active job at a time, lanes over its stages / template edges
            for (int i = 0; i < n_active; i++) {
                const int j = act[i];
                const JobRec &J = jb[j];
                const uint64_t active = J.active, sched = J.sched;
                const int nbase = dag_ptr[i], ns = J.n_stages;
                for (int s = lane; s < ns; s += 32) {
                    if (active & bit64(s)) {
                        const StageRec r = st[J.node_base + s];
                        int rank = nbase + popc64(active & (bit64(s) - 1));
                        nodes[rank * 3 + 0] = (float)r.remaining;
                        nodes[rank * 3 + 1] = r.mrd;
                        nodes[rank * 3 + 2] = (sched & bit64(s)) ? 1.0f : 0.0f;
                    }
                }
                const int eb = p.b_edge_base[J.tmpl], ne = p.b_edge_base[J.tmpl + 1] - eb;
                for (int k0 = 0; k0 < ne; k0 += 32) {
                    int k = k0 + lane, u = 0, v = 0;
                    bool keep = false;
                    if (k < ne) {
                        u = p.b_edges[2 * (eb + k)];
                        v = p.b_edges[2 * (eb + k) + 1];
                        keep = (active & bit64(u)) && (active & bit64(v));
                    }
                    unsigned m = __ballot_sync(FULL, keep);
                    if (keep) {
                        int pos = M + __popc(m & ((1u << lane) - 1));
                        edges[2 * pos] = nbase + popc64(active & (bit64(u) - 1));
                        edges[2 * pos + 1] = nbase + popc64(active & (bit64(v) - 1));
                    }
                    M += __popc(m);
                }
            }
        }
        if ((PARTS & OBS_HDR) && lane == 0) {
            ssb_obs_hdr o;
            o.reward = reward;
            o.wall_time = h->wall_time;
            o.num_nodes = N; o.num_edges = M; o.num_active_jobs = n_active;
            o.num_committable_execs = num_committable();
            o.source_job_idx = src_idx;
            o.num_schedulable = h->n_sched;
            o.error = h->error;
            o.terminated = terminated ? 1 : 0;
            o.truncated = (h->wall_time >= h->time_limit) ? 1 : 0;
            o.pending = 0; o.was_reset = 0;
            *oh = o;
            stats->observations++;
            stats->sum_nodes += N; stats->sum_edges += M; stats->sum_jobs += n_active;
        }
        __syncwarp();
    }

    // ------------------------------------------------------------ _take_action (:275-315), lane 0
    // returns 1: round finished (advance the simulation), 0: same round continues, -1: rejected
    __device__ int take_action(int stage_idx, int num_exec)
    {
        if (!(stage_idx >= -1 && stage_idx < oh->num_nodes && num_exec >= 1 && num_exec <= p.E))
            return -SSB_ENV_ACTION_SPACE;
        if (stage_idx == -1) {
            commit_remaining_executors();
            return (num_committable() > 0 && h->n_sched > 0) ? 0 : 1;
        }
        if (stage_idx >= h->n_sched) return -SSB_ENV_STAGE_KEY;
        // stage_selection_map[stage_idx]: the stage_idx-th schedulable stage in (job, stage) order
        int j = -1, s = -1, rem = stage_idx;
        for (int i = 0; i < h->n_active; i++) {
            uint64_t m = jb[act[i]].sched;
            int c = popc64(m);
            if (rem < c) {
                j = act[i];
                while (rem--) m &= m - 1;
                s = ffs64(m);
                break;
            }
            rem -= c;
        }
        if (j < 0) return -SSB_ENV_STAGE_KEY;
        if (num_exec > num_committable()) return -SSB_ENV_TOO_MANY_EXEC;
        const StageRec &r = st[jb[j].node_base + s];
        int demand = (int)r.remaining - ((int)r.moving_to + (int)r.commit_to);  // _adjust_num_executors
        int n = num_exec < demand ? num_exec : demand;
        if (n <= 0) { fail(1000 + __LINE__); return 1; }
        add_commitment(n, pool_of_stage(j, s));
        jb[j].selected |= bit64(s);
        // re-derive this job's schedulable stages only (bisect splice :306-315)
        int before = popc64(jb[j].sched);
        uint64_t m = job_sched_mask(j, source_job_id());
        jb[j].sched = m;
        h->n_sched += popc64(m) - before;
        return (num_committable() > 0 && h->n_sched > 0) ? 0 : 1;
    }

    // ------------------------------------------------------------ step() (:188-221)
    // max_events > 0 bounds the simulation work of this call: an environment that has not reached
    // its next decision yet is left "pending" (ssb_obs_hdr.pending = 1) and the next step_w() call on it
    // ignores its action arguments and simply continues.  max_events <= 0: reference semantics.
    // The pieces of step() before and after the simulation advances; step_w() strings them together.
    // step_begin_w: _take_action and, when the commitment round is over, its bookkeeping (:190-199).
    // Returns 0 when the step is already complete (same-round observation written, or the action was
    // rejected), 1 when the simulation has to advance.
    // DEFER (the fused rollout): observations are written as OBS_HDR only, and h->obs_owed is set to the parts of the
    // live observation that finish_obs_w still has to write (OWE_*); a rejected action leaves it as it is.  (In the
    // header rather than a register: a register live across the decision loop costs the one-slot kernel spills.)
    enum : int { OWE_GRAPH = 1, OWE_REWARD = 2 };
    template <bool DEFER = false>
    __device__ __forceinline__ int step_begin_w(int stage_idx, int num_exec)
    {
        SSB_T0();
        int rc = 0;
        if (lane == 0) rc = take_action(stage_idx, num_exec);
        rc = __shfl_sync(FULL, rc, 0);
        __syncwarp();
        if (rc < 0) {  // ValueError / KeyError: state untouched, report and let the caller retry
            if (lane == 0) oh->error = -rc;
            __syncwarp();
            return 0;
        }
        if (lane == 0) stats->decisions++;
        if (rc == 0) {
            SSB_TACC(5);
            if constexpr (DEFER) {  // reward 0: no time passed
                observe_w<OBS_HDR>(0.0, false);
                if (lane == 0) h->obs_owed = OWE_GRAPH;
            }
            else observe_w(0.0, false);
            SSB_TACC(7);
            return 0;
        }
        // commitment round has completed (:195-199)
        const int n_active0 = h->n_active;
        for (int i = lane; i < n_active0; i += 32) p.old_act[(size_t)b * p.Jc + i] = act[i];
        __syncwarp();
        if (lane == 0) {
            commit_remaining_executors();
            fulfill_commitments_from_source();
            h->source = POOL_NONE;
            h->wall_old = h->wall_time;
            h->n_old_active = n_active0;
        }
        __syncwarp();
        // selected_stages.clear() comes AFTER the fulfilment: backup scheduling during it must
        // still see this round's selections (:197-199, :825-839)
        for (int i = lane; i < n_active0; i += 32) jb[act[i]].selected = 0;
        __syncwarp();
        clear_sched_w();
        SSB_TACC(5);
        return 1;
    }
    // step_end_w: reward, termination flag and the next observation (:201-221)
    // (DEFER: the reward only when want_reward, else it is owed)
    template <bool DEFER = false>
    __device__ __forceinline__ void step_end_w(bool want_reward = true)
    {
        SSB_T0();
        double reward = 0.0;
        if (!DEFER || want_reward) reward = -compute_jobtime_w();
        bool terminated = false;
        if (lane == 0) {
            h->pending = 0;
            terminated = h->n_completed == h->n_jobs;
            if (terminated) { h->done = 1; stats->episodes++; }
            else if (!h->error && !(num_committable() > 0 && h->n_sched > 0)) fail(1000 + __LINE__);
        }
        terminated = __shfl_sync(FULL, (int)terminated, 0);
        __syncwarp();
        SSB_TACC(6);
        if constexpr (DEFER) {
            observe_w<OBS_HDR>(reward, terminated);
            if (lane == 0) h->obs_owed = want_reward ? OWE_GRAPH : OWE_GRAPH | OWE_REWARD;
        } else {
            observe_w(reward, terminated);
        }
        SSB_TACC(7);
    }
    // DEFER: see step_begin_w; only for max_events <= 0 (every call reaches its decision)
    template <int NS = 1, bool DEFER = false>
    __device__ void step_w(int stage_idx, int num_exec, int max_events = 0, bool want_reward = true)
    {
        if (h->error >= 1000) { if (lane == 0) oh->error = h->error; __syncwarp(); return; }
        if (h->done) { if (lane == 0) oh->error = SSB_ENV_DONE; __syncwarp(); return; }
        if (!h->pending) {
            if (step_begin_w<DEFER>(stage_idx, num_exec) == 0) return;
        }
        bool reached = true;
        if (!h->error) reached = resume_simulation_w<NS>(max_events);
        if (!reached) {
            if (lane == 0) {
                h->pending = 1;
                oh->pending = 1;
                oh->reward = 0.0;
                oh->wall_time = h->wall_time;
            }
            __syncwarp();
            return;
        }
        step_end_w<DEFER>(want_reward);
    }
    // the parts of the live observation a deferred step left owed (step_begin_w), written from the current state:
    // exact as long as nothing has changed the state since that step (compute_jobtime_w writes only its scratch)
    __device__ SSB_RARE void finish_obs_w()
    {
        SSB_T0();
        const int owed = h->obs_owed;
        if (owed & OWE_REWARD) {
            const double reward = -compute_jobtime_w();
            if (lane == 0) oh->reward = reward;
            __syncwarp();
        }
        if (owed & OWE_GRAPH) observe_w<OBS_GRAPH>(0.0, false);
        if (lane == 0) h->obs_owed = 0;
        __syncwarp();
        SSB_TACC(9);
    }

    // StochasticTimeLimit (wrappers/stochastic_time_limit.py:19-21): the episode's time limit ~ Exp(mean), drawn on
    // the Philox LIMIT stream of the episode's seed (oracle/philox_ref.py:time_limit_draw)
    __device__ double sample_time_limit(uint64_t seed) const
    {
        const uint4 w = philox4x32_10(0u, 0u, 3u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
        return __dmul_rn(p.mean_time_limit, neglog_u32(w.x));
    }
    // time limit of the episode an auto-reset starts: a fresh draw when a mean is configured, else unchanged
    __device__ double next_time_limit(uint64_t seed) const
    {
        return p.mean_time_limit > 0.0 ? sample_time_limit(seed) : h->time_limit;
    }

    // ------------------------------------------------------------ reset() (:127-186)
    __device__ SSB_RARE void reset_w(uint64_t seed, double time_limit)
    {
        const int Jc = p.Jc;
        int n_jobs = 0, err = 0;
        const bool trace = h->trace_jobs > 0;
        if (trace) {
            n_jobs = h->trace_jobs;
            for (int j = lane; j < n_jobs; j += 32) {
                jb[j].t_arrival = p.trace_t[(size_t)b * Jc + j];
                jb[j].tmpl = p.trace_tmpl[(size_t)b * Jc + j];
            }
        } else {
            // job_sequence (tpch.py:54-73) on the Philox job stream: draws in parallel, the running
            // sum of inter-arrival times sequentially (same f64 additions as `t += ...`)
            const int cap = p.job_arrival_cap;
            if (isinf(time_limit) && cap <= 0) err = SSB_ENV_NO_LIMIT;  // :137-138
            const int lim = cap > 0 ? min(cap, Jc) : Jc;
            for (int j = lane; j < lim; j += 32) {
                uint4 w = philox4x32_10((uint32_t)j, 0u, 1u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
                jb[j].tmpl = (int)bounded(w.y, 7) * 22 + (int)bounded(w.x, 22);  // tpch.py:177-178
                jb[j].t_completed = __dmul_rn(p.mean_interarrival, neglog_u32(w.z));  // stash x_j
            }
            __syncwarp();
            if (lane == 0 && !err) {
                double t = 0.0;
                int j = 0;
                while (t < time_limit && (cap <= 0 || j < cap)) {
                    if (j >= Jc) { err = SSB_ENV_CAPACITY; break; }
                    double x = jb[j].t_completed;
                    jb[j].t_arrival = t;
                    t = __dadd_rn(t, x);
                    j++;
                }
                n_jobs = j;
            }
            n_jobs = __shfl_sync(FULL, n_jobs, 0);
            err = __shfl_sync(FULL, err, 0);
        }
        __syncwarp();
        if (lane == 0) {
            int nb = 0, eb = 0;
            for (int j = 0; j < n_jobs; j++) {
                int t = jb[j].tmpl;
                jb[j].node_base = nb; jb[j].edge_base = eb;
                nb += p.b_num_stages[t];
                eb += p.b_edge_base[t + 1] - p.b_edge_base[t];
            }
            if (nb > p.Sc || eb > p.Mc) err = SSB_ENV_CAPACITY;
            EnvHdr &H = *h;
            H.wall_time = 0.0; H.time_limit = time_limit; H.wall_old = 0.0;
            H.seed = seed; H.log_n = 0; H.launch_idx = 0; H.seq = (uint32_t)n_jobs;
            H.n_jobs = n_jobs; H.next_arrival = 0; H.n_active = 0; H.n_completed = 0;
            H.source = POOL_COMMON; H.n_sched = 0; H.n_commits = 0; H.n_old_active = 0;
            H.commit_from_common = 0; H.commit_to_common = 0; H.total_none = 0;
            H.error = err; H.done = 0; H.n_nodes_total = nb; H.n_edges_total = eb;
            H.use_tape = (trace && H.tape_len >= 0) ? 1 : 0;
            H.pending = 0;
            H.policy_draws = 0;
            H.hist_n = 0;
            H.obs_owed = 0;
        }
        __syncwarp();
        if (h->error) {
            if (lane == 0) {
                ssb_obs_hdr o = {};
                o.error = h->error;
                *oh = o;
                if (h->error < 1000) { h->done = 1; }
            }
            __syncwarp();
            return;
        }
        // jobs
        for (int j = lane; j < n_jobs; j += 32) {
            JobRec &J = jb[j];
            int t = J.tmpl, ns = p.b_num_stages[t];
            J.ts_base = p.b_stage_base[t];
            J.n_stages = (int16_t)ns;
            J.t_completed = __longlong_as_double(0x7ff0000000000000ll);
            J.active = ns >= 64 ? ~0ull : (bit64(ns) - 1);
            uint64_t fr = 0;
            for (int s = 0; s < ns; s++)
                if (p.b_parent[J.ts_base + s] == 0) fr |= bit64(s);  // job.py:93-111 in-degree 0
            J.frontier = fr;
            J.sat = 0; J.sched = 0; J.selected = 0;
            J.n_local = 0; J.supply = 0; J.commit_from = 0; J.sat_count = 0; J.state = JOB_PENDING;
        }
        __syncwarp();
        // stages + their pools
        for (int j = 0; j < n_jobs; j++) {
            const JobRec &J = jb[j];
            for (int s = lane; s < J.n_stages; s += 32) {
                StageRec r;
                int nt = p.b_num_tasks[J.ts_base + s];
                r.remaining = (uint16_t)nt; r.completed = 0; r.num_tasks = (uint16_t)nt; r.job = (int16_t)j;
                r.commit_to = r.moving_to = r.commit_from = r.pad = 0;
                r.mrd = (float)p.b_rough[J.ts_base + s];
                st[J.node_base + s] = r;
            }
        }
        // pools: fresh `set()` everywhere (executor_tracker.py:39-42, :77, :90)
        const int n_pools = 2 + Jc + h->n_nodes_total;
        for (int q = lane; q < n_pools; q += 32) {
            PoolHdr hd; hd.mask = 7; hd.fill = 0; hd.used = 0; hd.finger = 0;
            ph[q] = hd;
            uint8_t *t = pt + (size_t)q * p.TAB;
            *reinterpret_cast<unsigned long long *>(t) = ~0ull;  // 8 EMPTY slots
        }
        for (int e = lane; e < p.E; e += 32) {
            ExecRec x = {};
            x.job_id = -1; x.task_stage = -1; x.loc = POOL_COMMON; x.ev_task = -1;
            ex[e] = x;
        }
        __syncwarp();
        if (lane == 0) {
            PSet<uint8_t> c = ps_load(POOL_COMMON);  // set(range(num_executors))
            for (int e = 0; e < p.E; e++) ps_add(c, e, scr + 2 * p.TAB);
            ps_store(POOL_COMMON, c);
            // _load_initial_jobs (:260-273): arrivals with t <= 0, wall_time stays 0
            while (h->next_arrival < n_jobs && jb[h->next_arrival].t_arrival <= 0.0)
                handle_job_arrival(h->next_arrival++);
        }
        __syncwarp();
        find_schedulable_all_w();
        observe_w(0.0, false);
    }

    // ------------------------------------------------------------ Decima observation adapter
    // DecimaObsWrapper.observation (schedulers/decima/env_wrapper.py:69-143): commit caps, the five
    // node features, stage mask; make_dag_layer_edge_masks (schedulers/decima/utils.py:238-267):
    // topological generations of the active graph, mask k = edges with both ends in L_k U succ(L_k),
    // emitted per edge as a bit set over k.  Jobs are disjoint DAGs, so generations are found per
    // job on u64 masks: L_k = active unassigned stages without an active unassigned parent.
    // Sk: per-warp shared scratch (>= 64 entries).
    __device__ SSB_RARE void decima_obs_w(uint64_t *Sk)
    {
        const int n_active = h->n_active, ncommit = num_committable(), src_job = source_job_id();
        float *feat = p.dec_feat + (size_t)b * p.Sc * 5;
        uint8_t *smask = p.dec_stage_mask + (size_t)b * p.Sc;
        uint8_t *fmask = p.dec_frontier_mask + (size_t)b * p.Sc;
        int32_t *caps = p.dec_caps + (size_t)b * p.Jc;
        uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
        const double Ed = (double)p.E;
        int N = 0, M = 0, D = 0;
        for (int i = 0; i < n_active; i++) {
            const int j = act[i];
            const JobRec &J = jb[j];
            const uint64_t active = J.active, sched = J.sched, frontier = J.frontier;
            const int supply = J.supply, ns = J.n_stages;
            int cap = min(max(p.E - supply, 0), ncommit);  // :74-77
            if (j == src_job) cap = ncommit;               // :81-82
            if (lane == 0) caps[i] = cap;
            const float f0 = (float)((double)cap / Ed), f1 = (j == src_job) ? 1.0f : -1.0f,
                        f2 = (float)((double)supply / Ed);
            for (int s = lane; s < ns; s += 32) {
                if (!((active >> s) & 1)) continue;
                const StageRec r = st[J.node_base + s];
                const int rank = N + popc64(active & (bit64(s) - 1));
                const float rem = (float)r.remaining;
                float *f = feat + (size_t)rank * 5;
                f[0] = f0; f[1] = f1; f[2] = f2;
                f[3] = __fdiv_rn(rem, 200.0f);                          // float32 / num_tasks_scale (:137)
                f[4] = __fdiv_rn(__fmul_rn(rem, r.mrd), 100000.0f);     // float32 * float32 / work_scale (:141)
                smask[rank] = (uint8_t)((sched >> s) & 1);
                fmask[rank] = (uint8_t)((frontier >> s) & 1);
            }
            const uint64_t *pm = p.b_parent + J.ts_base, *cm = p.b_child + J.ts_base;
            const int eb = p.b_edge_base[J.tmpl], ne = p.b_edge_base[J.tmpl + 1] - eb;
            int dj = 0;
            if (ns <= 32) {
                // Jobs of up to 32 stages (every TPC-H template): 32-bit masks, one stage per lane.  Lane s keeps
                // the set of levels k with s in L_k U succ(L_k) in a register; an edge's mask bits are then the
                // AND of its two ends' level sets (read through shared memory).
                const uint32_t act32 = (uint32_t)active;
                const uint32_t pm32 = lane < ns ? (uint32_t)pm[lane] : 0u, cm32 = lane < ns ? (uint32_t)cm[lane] : 0u;
                uint32_t assigned = 0;
                uint64_t ls = 0;
                while (assigned != act32 && dj < 64) {
                    const uint32_t open = act32 & ~assigned;
                    const bool r0 = ((open >> lane) & 1) && (pm32 & open) == 0;
                    const uint32_t Lk = __ballot_sync(FULL, r0);
                    const uint32_t S = Lk | __reduce_or_sync(FULL, r0 ? (cm32 & act32) : 0u);
                    if ((S >> lane) & 1) ls |= bit64(dj);
                    assigned |= Lk;
                    dj++;
                    if (Lk == 0) break;  // cannot happen in a DAG
                }
                Sk[lane] = ls;
                __syncwarp();
                for (int k0 = 0; k0 < ne; k0 += 32) {
                    const int k = k0 + lane;
                    int u = 0, v = 0;
                    bool keep = false;
                    if (k < ne) {
                        u = p.b_edges[2 * (eb + k)];
                        v = p.b_edges[2 * (eb + k) + 1];
                        keep = ((act32 >> u) & 1) && ((act32 >> v) & 1);
                    }
                    const unsigned m = __ballot_sync(FULL, keep);
                    if (keep) ebits[M + __popc(m & ((1u << lane) - 1))] = Sk[u] & Sk[v];
                    M += __popc(m);
                }
            } else {
                uint64_t assigned = 0;
                while (assigned != active && dj < 64) {
                    const uint64_t open = active & ~assigned;
                    const int s0 = lane, s1 = lane + 32;
                    const bool r0 = s0 < ns && ((open >> s0) & 1) && (pm[s0] & open) == 0;
                    const bool r1 = s1 < ns && ((open >> s1) & 1) && (pm[s1] & open) == 0;
                    const uint64_t Lk = (uint64_t)__ballot_sync(FULL, r0) | ((uint64_t)__ballot_sync(FULL, r1) << 32);
                    const uint64_t mine = ((r0 ? cm[s0] : 0ull) | (r1 ? cm[s1] : 0ull)) & active;
                    const uint64_t succ = (uint64_t)__reduce_or_sync(FULL, (uint32_t)mine) |
                                          ((uint64_t)__reduce_or_sync(FULL, (uint32_t)(mine >> 32)) << 32);
                    if (lane == 0) Sk[dj] = Lk | succ;
                    assigned |= Lk;
                    dj++;
                    if (Lk == 0) break;  // cannot happen in a DAG
                }
                __syncwarp();
                for (int k0 = 0; k0 < ne; k0 += 32) {
                    const int k = k0 + lane;
                    int u = 0, v = 0;
                    bool keep = false;
                    if (k < ne) {
                        u = p.b_edges[2 * (eb + k)];
                        v = p.b_edges[2 * (eb + k) + 1];
                        keep = ((active >> u) & 1) && ((active >> v) & 1);
                    }
                    const unsigned m = __ballot_sync(FULL, keep);
                    if (keep) {
                        uint64_t bits = 0;
                        for (int q = 0; q < dj; q++) {
                            const uint64_t S = Sk[q];
                            if (((S >> u) & 1) && ((S >> v) & 1)) bits |= bit64(q);
                        }
                        ebits[M + __popc(m & ((1u << lane) - 1))] = bits;
                    }
                    M += __popc(m);
                }
            }
            D = max(D, dj);
            __syncwarp();
            N += popc64(active);
        }
        if (lane == 0) p.dec_depth[b] = D > 1 ? D - 1 : 0;
    }

    // ------------------------------------------------------------ fair / FIFO policy
    // RoundRobinScheduler.schedule (schedulers/heuristics/round_robin.py:14-49) with
    // preprocess_obs/find_stage (heuristics/utils.py:5-37).  "Frontier" there means "no incoming
    // edge in the observed sub-graph", i.e. every parent completed == Job.frontier_stages.
    __device__ void fair_action_w(bool dynamic_partition, int &stage_idx, int &num_exec)
    {
        const int Ja = h->n_active, ncommit = num_committable();
        const int src_job = source_job_id();
        const int cap = dynamic_partition ? (p.E + max(1, Ja) - 1) / max(1, Ja) : p.E;
        int best_n = ncommit, run = 0, best_rank = -1;
        for (int base = 0; base < Ja; base += 32) {
            int i = base + lane, j = -1, cnt = 0, sel = -1, supply = 0;
            uint64_t m = 0;
            if (i < Ja) {
                j = act[i];
                m = jb[j].sched;
                cnt = popc64(m);
                supply = jb[j].supply;
                if (m) {  // find_stage: first schedulable frontier stage, else first schedulable
                    uint64_t f = m & jb[j].frontier;
                    sel = ffs64(f ? f : m);
                }
            }
            int incl = cnt;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                int v = __shfl_up_sync(FULL, incl, off);
                if (lane >= off) incl += v;
            }
            int rank = sel >= 0 ? run + incl - cnt + popc64(m & (bit64(sel) - 1)) : -1;
            bool is_src = j >= 0 && j == src_job;
            unsigned srcb = __ballot_sync(FULL, is_src);
            if (srcb) {
                int l = __ffs(srcb) - 1;
                int r = __shfl_sync(FULL, rank, l);
                if (r >= 0) { stage_idx = r; num_exec = ncommit; return; }  // source job first
            }
            bool ok = (i < Ja) && !is_src && supply < cap && sel >= 0;
            unsigned okb = __ballot_sync(FULL, ok);
            if (okb && best_rank < 0) {
                int l = __ffs(okb) - 1;
                best_rank = __shfl_sync(FULL, rank, l);
                int sp = __shfl_sync(FULL, supply, l);
                best_n = min(ncommit, cap - sp);
            }
            run += __shfl_sync(FULL, incl, 31);
        }
        if (best_rank >= 0) { stage_idx = best_rank; num_exec = best_n; return; }
        stage_idx = -1;
        num_exec = ncommit;
    }

#ifdef SSB_RANDOM_POLICY
    // ------------------------------------------------------------ random policy
    // (compiled only in ssb_random.cu, so that the simulator's translation unit is unchanged)
    // RandomScheduler.schedule (schedulers/heuristics/random_scheduler.py:7-32) in law: the reference redraws a job
    // uniformly from the jobs still "running" until find_stage gives a stage, i.e. one uniform draw over the active
    // jobs that have a schedulable stage ("eligible"); num_exec ~ U[1, num_committable].  Draws: the RANDOM stream,
    // Philox ctr (policy_draws, 0, 5, 0), key = episode seed (tests/random_policy_spec.py); every call
    // advances policy_draws, also when no job is eligible (stage_idx = -1).
    __device__ void random_action_w(int &stage_idx, int &num_exec)
    {
        const int Ja = h->n_active, ncommit = num_committable();
        const uint32_t pd = h->policy_draws;
        int k = 0;  // eligible jobs
#pragma unroll 1  // (both loops: unrolled, they cost the one-slot rollout kernel spills)
        for (int base = 0; base < Ja; base += 32) {
            const int i = base + lane;
            k += __popc(__ballot_sync(FULL, i < Ja && jb[act[i]].sched != 0));
        }
        const uint4 w = philox4x32_10(pd, 0u, 5u, 0u, (uint32_t)h->seed, (uint32_t)(h->seed >> 32));
        const int t = (int)bounded(w.x, (uint32_t)k);  // the t-th eligible job in active-job order
        num_exec = 1 + (int)bounded(w.y, (uint32_t)max(ncommit, 0));
        stage_idx = -1;
        int run = 0, seen = 0;  // schedulable stages / eligible jobs before this chunk
#pragma unroll 1
        for (int base = 0; base < Ja && k > 0; base += 32) {
            const int i = base + lane;
            uint64_t m = 0;
            int below = 0;  // schedulable stages of this job before its find_stage choice
            bool el = false;
            if (i < Ja) {
                const int j = act[i];
                m = jb[j].sched;
                if (m) {  // find_stage: first schedulable frontier stage, else first schedulable
                    const uint64_t f = m & jb[j].frontier;
                    below = popc64(m & (bit64(ffs64(f ? f : m)) - 1));
                    el = true;
                }
            }
            const unsigned eb = __ballot_sync(FULL, el);
            if (t < seen + __popc(eb)) {
                const int l = __fns(eb, 0, t - seen + 1);  // lane of the (t - seen)-th eligible job of the chunk
                run += (int)__reduce_add_sync(FULL, lane < l ? (unsigned)popc64(m) : 0u);
                stage_idx = run + __shfl_sync(FULL, below, l);
                break;
            }
            seen += __popc(eb);
            run += (int)__reduce_add_sync(FULL, (unsigned)popc64(m));
        }
        __syncwarp();
        if (lane == 0) h->policy_draws = pd + 1;
        __syncwarp();
    }
#endif

#ifdef SSB_DECIMA_CTA_ADAPTER
    // ------------------------------------------------------------ Decima adapter, one CTA per environment
    // (k_decima_obs_cta, ssb_policy.cu; compiled only there so that the simulator's translation unit is unchanged).
    // decima_obs_w walks the active jobs one after the other -- a chain of dependent loads per job that one warp
    // cannot hide.  Here the jobs' node offsets come from the observation's dag_ptr, their edge offsets from a count
    // pass with one THREAD per job, and the warps of the CTA then take the jobs round-robin.
    // what pass 2 needs of a job, fetched by pass 1 (one thread per job) into shared memory: the per-job chain of
    // dependent loads (active list -> job record -> template -> edges) then runs for all jobs at once
    struct AdJob { uint64_t active, sched, frontier; int32_t supply, ns, node_base, ts_base, eb, ne, j, n_edges; };
    // pass 1 for the i-th active job; n_edges = its edges that stay in the observation (both ends active),
    // utils.subgraph (utils.py:5-22)
    __device__ AdJob decima_job_fetch(int i) const
    {
        AdJob a;
        a.j = act[i];
        const JobRec &J = jb[a.j];
        a.active = J.active; a.sched = J.sched; a.frontier = J.frontier;
        a.supply = J.supply; a.ns = J.n_stages; a.node_base = J.node_base; a.ts_base = J.ts_base;
        a.eb = p.b_edge_base[J.tmpl];
        a.ne = p.b_edge_base[J.tmpl + 1] - a.eb;
        a.n_edges = job_obs_edges(a.active, a.eb, a.ne);
        return a;
    }
    // the i-th active job's share of decima_obs_w (env_wrapper.py:69-143, decima/utils.py:238-267): node rows N..,
    // edge entries M..; returns the number of topological generations of the job's active sub-graph
    __device__ int decima_obs_job_w(const AdJob &A, int i, int N, int M, int ncommit, int src_job, uint64_t *Sk)
    {
        float *feat = p.dec_feat + (size_t)b * p.Sc * 5;
        uint8_t *smask = p.dec_stage_mask + (size_t)b * p.Sc;
        uint8_t *fmask = p.dec_frontier_mask + (size_t)b * p.Sc;
        uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
        const double Ed = (double)p.E;
        const int j = A.j;
        const uint64_t active = A.active, sched = A.sched, frontier = A.frontier;
        const int supply = A.supply, ns = A.ns;
        int cap = min(max(p.E - supply, 0), ncommit);  // :74-77
        if (j == src_job) cap = ncommit;               // :81-82
        if (lane == 0) p.dec_caps[(size_t)b * p.Jc + i] = cap;
        // float32(cap / E) as the reference computes it in double and stores in float32: for integers 0 <= cap <= E
        // <= 128 the float32 division gives the same bits (checked exhaustively, tests/test_decima_obs_oracle.py),
        // and it avoids two software fp64 divisions per job (9 % of this kernel's instructions)
        const float f0 = __fdiv_rn((float)cap, (float)p.E), f1 = (j == src_job) ? 1.0f : -1.0f;
        const float f2 = supply <= p.E ? __fdiv_rn((float)supply, (float)p.E) : (float)((double)supply / Ed);
        for (int s = lane; s < ns; s += 32) {
            if (!((active >> s) & 1)) continue;
            const StageRec r = st[A.node_base + s];
            const int rank = N + popc64(active & (bit64(s) - 1));
            const float rem = (float)r.remaining;
            float *f = feat + (size_t)rank * 5;
            f[0] = f0; f[1] = f1; f[2] = f2;
            f[3] = __fdiv_rn(rem, 200.0f);                       // float32 / num_tasks_scale (:137)
            f[4] = __fdiv_rn(__fmul_rn(rem, r.mrd), 100000.0f);  // float32 * float32 / work_scale (:141)
            smask[rank] = (uint8_t)((sched >> s) & 1);
            fmask[rank] = (uint8_t)((frontier >> s) & 1);
        }
        const uint64_t *pm = p.b_parent + A.ts_base, *cm = p.b_child + A.ts_base;
        const int eb = A.eb, ne = A.ne;
        int dj = 0;
        if (ns <= 32) {  // one stage per lane, level sets in registers (see decima_obs_w)
            const uint32_t act32 = (uint32_t)active;
            const uint32_t pm32 = lane < ns ? (uint32_t)pm[lane] : 0u, cm32 = lane < ns ? (uint32_t)cm[lane] : 0u;
            uint32_t assigned = 0;
            uint64_t ls = 0;
            while (assigned != act32 && dj < 64) {
                const uint32_t open = act32 & ~assigned;
                const bool r0 = ((open >> lane) & 1) && (pm32 & open) == 0;
                const uint32_t Lk = __ballot_sync(FULL, r0);
                const uint32_t S = Lk | __reduce_or_sync(FULL, r0 ? (cm32 & act32) : 0u);
                if ((S >> lane) & 1) ls |= bit64(dj);
                assigned |= Lk;
                dj++;
                if (Lk == 0) break;  // cannot happen in a DAG
            }
            Sk[lane] = ls;
            __syncwarp();
            for (int k0 = 0; k0 < ne; k0 += 32) {
                const int k = k0 + lane;
                int u = 0, v = 0;
                bool keep = false;
                if (k < ne) {
                    u = p.b_edges[2 * (eb + k)];
                    v = p.b_edges[2 * (eb + k) + 1];
                    keep = ((act32 >> u) & 1) && ((act32 >> v) & 1);
                }
                const unsigned m = __ballot_sync(FULL, keep);
                if (keep) ebits[M + __popc(m & ((1u << lane) - 1))] = Sk[u] & Sk[v];
                M += __popc(m);
            }
        } else {
            uint64_t assigned = 0;
            while (assigned != active && dj < 64) {
                const uint64_t open = active & ~assigned;
                const int s0 = lane, s1 = lane + 32;
                const bool r0 = s0 < ns && ((open >> s0) & 1) && (pm[s0] & open) == 0;
                const bool r1 = s1 < ns && ((open >> s1) & 1) && (pm[s1] & open) == 0;
                const uint64_t Lk = (uint64_t)__ballot_sync(FULL, r0) | ((uint64_t)__ballot_sync(FULL, r1) << 32);
                const uint64_t mine = ((r0 ? cm[s0] : 0ull) | (r1 ? cm[s1] : 0ull)) & active;
                const uint64_t succ = (uint64_t)__reduce_or_sync(FULL, (uint32_t)mine) |
                                      ((uint64_t)__reduce_or_sync(FULL, (uint32_t)(mine >> 32)) << 32);
                if (lane == 0) Sk[dj] = Lk | succ;
                assigned |= Lk;
                dj++;
                if (Lk == 0) break;
            }
            __syncwarp();
            for (int k0 = 0; k0 < ne; k0 += 32) {
                const int k = k0 + lane;
                int u = 0, v = 0;
                bool keep = false;
                if (k < ne) {
                    u = p.b_edges[2 * (eb + k)];
                    v = p.b_edges[2 * (eb + k) + 1];
                    keep = ((active >> u) & 1) && ((active >> v) & 1);
                }
                const unsigned m = __ballot_sync(FULL, keep);
                if (keep) {
                    uint64_t bits = 0;
                    for (int q = 0; q < dj; q++) {
                        const uint64_t S = Sk[q];
                        if (((S >> u) & 1) && ((S >> v) & 1)) bits |= bit64(q);
                    }
                    ebits[M + __popc(m & ((1u << lane) - 1))] = bits;
                }
                M += __popc(m);
            }
        }
        __syncwarp();
        return dj;
    }
#endif
};

}  // namespace ssb
