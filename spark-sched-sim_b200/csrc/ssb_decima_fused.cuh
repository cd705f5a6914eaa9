// ssb_decima_fused.cuh -- the Decima policy's three-layer MLPs on the 5th-generation tensor cores with the
// activations kept in TENSOR MEMORY between layers (tcgen05.mma with the A operand in TMEM), and fp32 accuracy
// from bf16 hardware by a three-way operand split.
//
// A 128-row tile is owned by one warpgroup (thread r <-> tile row r <-> TMEM lane r):
//   gather 128 input rows -> split -> tcgen05.st into TMEM (A operand)
//   layer: one elected thread issues tcgen05.mma.kind::f16 (A from TMEM, W from shared memory, D in TMEM),
//          tcgen05.commit -> mbarrier; every thread reads its row of D back with tcgen05.ld, adds the bias,
//          applies the activation in fp32 registers, splits again and tcgen05.st's the next layer's A operand
//   last layer's row -> scatter.
// Nothing but the (small, read-only) weights lives in shared memory: the round-1 kernel wrote every layer's A tile
// to shared memory (hi + lo, 64 KB per tile) and the tensor core read ~110 KB of operands per tile back from it --
// the shared-memory pipe was the bound (profiles/r01_ncu_k_tile_mlp_mid_episode.csv).  TMEM columns per warpgroup:
// D at [0, 32), the three split terms of A at [32 + 32 j, 32 + 32 j + K / 2), j = 0..2 (two bf16 per 32-bit column).
//
// fp32 accuracy: x = b0 + b1 + b2 EXACTLY, each term a bf16 (8 significant bits: 8 + 8 + 8 = the 24 of an fp32),
// same for the weights; a product is accumulated as eight of the nine partial products (smallest first, fp32
// accumulation in TMEM); the dropped b2 * w2 is below 2^-30 relative.  The activations are split by TRUNCATION (the
// three bytes of the significand: one AND + one subtraction per term, packing by byte permute straight from the
// remainders -- 5.5 ALU instructions per element), the weights once per upload by rounding.  Measured against an fp64
// evaluation of the reference's model: tests/test_gpu_decima_policy.py::test_mlp_rows_accuracy_against_fp64.
#pragma once
#include "ssb_decima_tc.cuh"

namespace ssb {
namespace fz {

using tc::fence_async_smem;
using tc::mbar_init;
using tc::mbar_wait;
using tc::smem_u32;
using tc::tc_fence_after;
using tc::tc_fence_before;
using tc::tmem_alloc;
using tc::tmem_dealloc;
using tc::umma_commit;
using tc::umma_desc;

// instruction descriptor (cute::UMMA::InstrDescriptor): D = f32, A = B = bf16, both K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N)
{
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[tmem] . B[smem]^T, one instruction = K 16
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t *r)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
                 "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// x = b0 + b1 + b2 exactly (each term a bf16 held in the upper half of a 32-bit pattern).  b0, b1: nearest (ties away
// from zero, on the integer ALU); the remainder after two steps has at most 8 significant bits, so b2 is exact.
__device__ __forceinline__ void split3(float x, uint32_t &b0, uint32_t &b1, uint32_t &b2)
{
    b0 = (__float_as_uint(x) + 0x8000u) & 0xffff0000u;
    const float r1 = x - __uint_as_float(b0);
    b1 = (__float_as_uint(r1) + 0x8000u) & 0xffff0000u;
    b2 = __float_as_uint(r1 - __uint_as_float(b1));
}
// two bf16 (upper halves of lo / hi) in one 32-bit TMEM column: element k (even) in the low half, k + 1 in the high
__device__ __forceinline__ uint32_t pack2(uint32_t lo, uint32_t hi) { return __byte_perm(lo, hi, 0x7632); }

// ------------------------------------------------------------------ the seven MLPs
// K0: input width padded to the MMA's K granularity (16); IN: real input width; W: offset in the dd weight layout
template <int ST> struct Spec;
template <> struct Spec<tc::ST_PREP>  { static constexpr int K0 = 16, IN = 5,  H1 = 32, H2 = 16, OUT = 16, W = dd::PREP;  static constexpr bool TANH = false; };
template <> struct Spec<tc::ST_SINK>  { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::UPD;   static constexpr bool TANH = false; };
template <> struct Spec<tc::ST_MSG>   { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::MSG;   static constexpr bool TANH = false; };
template <> struct Spec<tc::ST_RCV>   { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::UPD;   static constexpr bool TANH = false; };
template <> struct Spec<tc::ST_DAG>   { static constexpr int K0 = 32, IN = 21, H1 = 32, H2 = 16, OUT = 16, W = dd::DAG;   static constexpr bool TANH = false; };
template <> struct Spec<tc::ST_GLOB>  { static constexpr int K0 = 16, IN = 16, H1 = 32, H2 = 16, OUT = 16, W = dd::GLOB;  static constexpr bool TANH = false; };
template <> struct Spec<tc::ST_STAGE> { static constexpr int K0 = 64, IN = 53, H1 = 64, H2 = 64, OUT = 1,  W = dd::STAGE; static constexpr bool TANH = true; };
template <> struct Spec<tc::ST_EXEC>  { static constexpr int K0 = 48, IN = 36, H1 = 64, H2 = 64, OUT = 1,  W = dd::EXEC;  static constexpr bool TANH = true; };

// A stage's constant "weight blob" (built once per weight upload, copied to shared memory as is), in 4-byte words:
//   layer 1: three bf16 tiles [H1 x K0] (split terms 0, 1, 2), canonical K-major no-swizzle UMMA layout
//            (8-row x 16-byte core matrices: 8 bf16 along K; LBO = 128 B between K chunks, SBO = K * 16 B between
//            8-row groups); layer 2: three tiles [H2 x H1]; layer 3 (OUT > 1): three tiles [OUT x H2];
//   then fp32: biases (H1 + H2 + max(OUT, 1)), and for OUT == 1 the last layer's H2 weights.
template <int ST>
struct Blob {
    using S = Spec<ST>;
    static constexpr int W1 = 0;                                   // words
    static constexpr int W2 = W1 + 3 * S::H1 * S::K0 / 2;
    static constexpr int W3 = W2 + 3 * S::H2 * S::H1 / 2;
    static constexpr int BIAS = W3 + (S::OUT > 1 ? 3 * S::OUT * S::H2 / 2 : 0);
    static constexpr int W3V = BIAS + S::H1 + S::H2 + 16;
    static constexpr int WORDS = (W3V + (S::OUT > 1 ? 0 : S::H2) + 3) & ~3;
};
__host__ __device__ constexpr int blob3_words(int st)
{
    return st == tc::ST_PREP ? Blob<tc::ST_PREP>::WORDS : st == tc::ST_SINK ? Blob<tc::ST_SINK>::WORDS
         : st == tc::ST_MSG ? Blob<tc::ST_MSG>::WORDS : st == tc::ST_RCV ? Blob<tc::ST_RCV>::WORDS
         : st == tc::ST_DAG ? Blob<tc::ST_DAG>::WORDS : st == tc::ST_GLOB ? Blob<tc::ST_GLOB>::WORDS
         : st == tc::ST_STAGE ? Blob<tc::ST_STAGE>::WORDS : Blob<tc::ST_EXEC>::WORDS;
}
__host__ __device__ constexpr int blob3_offset(int st)
{
    int off = 0;
    for (int i = 0; i < st; i++) off += blob3_words(i);
    return off;
}
constexpr int BLOB_TOTAL = blob3_offset(tc::ST_EXEC) + blob3_words(tc::ST_EXEC);

// bf16 element offset of (row n, k) in a canonical [rows x K] tile
__host__ __device__ __forceinline__ int canon16(int n, int k, int K)
{
    return (n >> 3) * (K * 8) + (k >> 3) * 64 + (n & 7) * 8 + (k & 7);
}
// dd-layout Linear (transposed weight [in][out], then the bias) -> three canonical bf16 tiles + the bias
template <int IN, int K, int N>
__device__ __forceinline__ void build_layer(const float *__restrict__ wt, uint16_t *tiles, float *bias, int tid, int nthr)
{
    for (int i = tid; i < N * K; i += nthr) {
        const int n = i / K, k = i % K;
        const float x = k < IN ? wt[k * N + n] : 0.0f;
        uint32_t b0, b1, b2;
        split3(x, b0, b1, b2);
        const int off = canon16(n, k, K);
        tiles[off] = (uint16_t)(b0 >> 16);
        tiles[N * K + off] = (uint16_t)(b1 >> 16);
        tiles[2 * N * K + off] = (uint16_t)(b2 >> 16);
    }
    for (int i = tid; i < N; i += nthr) bias[i] = wt[dd::pad4(IN * N) + i];
}
template <int ST>
__global__ void __launch_bounds__(128) k_build_blob(const float *pol_w, uint32_t *blob_all)
{
    using S = Spec<ST>;
    using L = Blob<ST>;
    uint32_t *bl = blob_all + blob3_offset(ST);
    float *bias = reinterpret_cast<float *>(bl + L::BIAS);
    const float *w = pol_w + S::W;
    const int tid = threadIdx.x;
    build_layer<S::IN, S::K0, S::H1>(w, reinterpret_cast<uint16_t *>(bl + L::W1), bias, tid, 128);
    build_layer<S::H1, S::H1, S::H2>(w + dd::layer(S::IN, S::H1), reinterpret_cast<uint16_t *>(bl + L::W2), bias + S::H1,
                                     tid, 128);
    const float *w3 = w + dd::layer(S::IN, S::H1) + dd::layer(S::H1, S::H2);
    if constexpr (S::OUT > 1) {
        build_layer<S::H2, S::H2, S::OUT>(w3, reinterpret_cast<uint16_t *>(bl + L::W3), bias + S::H1 + S::H2, tid, 128);
    } else {
        float *w3v = reinterpret_cast<float *>(bl + L::W3V);
        for (int i = tid; i < S::H2; i += 128) w3v[i] = w3[i];  // [H2][1], then the bias
        if (tid == 0) bias[S::H1 + S::H2] = w3[dd::pad4(S::H2)];
    }
}

// ------------------------------------------------------------------ one warpgroup's tile context
struct Wg {
    uint32_t tmem;    // this warpgroup's 128 TMEM columns (lane 0)
    uint32_t trow;    // ... seen from this thread's warp (lane field = 32 * (warp % 4))
    uint32_t mbar;    // its mbarrier (shared-memory address)
    uint32_t parity;
    int tid;          // 0..127 within the warpgroup
    int bar;          // named barrier id of the warpgroup
};
// TMEM column maps of one tile context.  128 columns: D at [0, 32), A term j at [32 + 32 j, ...).  64 columns (the
// 16-wide GNN MLPs): D at [0, N), the three A terms packed at the top, [64 - 3 K / 2, 64) -- layer 1 (N 32, K 16): D
// [0, 32) A [40, 64); layer 2 (N 16, K 32): D [0, 16) A [16, 64); layer 3: D [0, 16) A [40, 64).  A thread only ever
// reads and writes its OWN lane, and a layer's A is written after the previous layer's D was read into registers
// and its MMAs have completed, so the regions of consecutive layers may overlap.
constexpr int COL_D = 0, COLS_PER_WG = 128;
template <int COLS, int K> __device__ __forceinline__ constexpr int a_base() { return COLS == 64 ? 64 - 3 * K / 2 : 32; }
template <int COLS, int K> __device__ __forceinline__ constexpr int a_stride() { return COLS == 64 ? K / 2 : 32; }

__device__ __forceinline__ void wg_sync(const Wg &g) { asm volatile("bar.sync %0, 128;" ::"r"(g.bar) : "memory"); }

// this thread's row of the next layer's A operand: v[0..K) -> three bf16 terms, two per column
template <int K, int COLS = 128>
__device__ __forceinline__ void store_a_row(const Wg &g, const float *v)
{
    // truncation split: term j = the j-th byte of the significand (x & 0xffff0000 is a bf16; x minus it is exact);
    // pack2 takes the upper halves straight from x, the first and the second remainder
#pragma unroll
    for (int c0 = 0; c0 < K / 2; c0 += 8) {
        uint32_t t0[8], t1[8], t2[8];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const float x0 = v[2 * (c0 + c)], x1 = v[2 * (c0 + c) + 1];
            const float r0 = x0 - __uint_as_float(__float_as_uint(x0) & 0xffff0000u);
            const float r1 = x1 - __uint_as_float(__float_as_uint(x1) & 0xffff0000u);
            const float s0 = r0 - __uint_as_float(__float_as_uint(r0) & 0xffff0000u);
            const float s1 = r1 - __uint_as_float(__float_as_uint(r1) & 0xffff0000u);
            t0[c] = pack2(__float_as_uint(x0), __float_as_uint(x1));
            t1[c] = pack2(__float_as_uint(r0), __float_as_uint(r1));
            t2[c] = pack2(__float_as_uint(s0), __float_as_uint(s1));
        }
        tmem_st8(g.trow + a_base<COLS, K>() + c0, t0);
        tmem_st8(g.trow + a_base<COLS, K>() + a_stride<COLS, K>() + c0, t1);
        tmem_st8(g.trow + a_base<COLS, K>() + 2 * a_stride<COLS, K>() + c0, t2);
    }
    tmem_wait_st();
}
// D[128 x N] = A[128 x K] . W[n0 .. n0 + N)[K]^T : eight partial products a_i * w_j (all but a_2 * w_2), smallest first.
// w = the layer's three tiles in shared memory (term j at w + j * NTOT * K bf16).  One elected thread.
template <int K, int N, int NTOT, int COLS = 128>
__device__ __forceinline__ void issue_layer(const Wg &g, const uint32_t *w_words, int n0)
{
    constexpr uint32_t idesc = umma_idesc_bf16(128, N);
    constexpr uint32_t sbo = K * 16;
    constexpr uint32_t term_bytes = NTOT * K * 2;
    // one descriptor for the layer's first tile; the other terms / k-steps differ in the start-address field only
    const uint64_t d0 = umma_desc(smem_u32(w_words) + (uint32_t)(n0 >> 3) * sbo, 128, sbo);
    const uint32_t a0 = g.tmem + a_base<COLS, K>();
    const int ai[8] = {2, 1, 2, 0, 1, 1, 0, 0}, wi[8] = {1, 2, 0, 2, 1, 0, 1, 0};
    bool first = true;
#pragma unroll
    for (int q = 0; q < 8; q++) {
#pragma unroll
        for (int ks = 0; ks < K / 16; ks++) {
            umma_bf16_ts(g.tmem + COL_D, a0 + a_stride<COLS, K>() * ai[q] + ks * 8,
                         d0 + (uint64_t)((wi[q] * term_bytes + ks * 256) >> 4), idesc, first ? 0u : 1u);
            first = false;
        }
    }
    umma_commit(g.mbar);
}
// A written by every thread -> MMAs issued -> D complete and visible to every thread of the warpgroup
template <int K, int N, int NTOT, int COLS = 128>
__device__ __forceinline__ void run_layer(Wg &g, const uint32_t *w_words, int n0)
{
    tc_fence_before();
    wg_sync(g);
    if (g.tid == 0) {
        tc_fence_after();
        issue_layer<K, N, NTOT, COLS>(g, w_words, n0);
    }
    mbar_wait(g.mbar, g.parity);
    g.parity ^= 1;
    tc_fence_after();
}

template <bool TANH>
__device__ __forceinline__ float act(float x)
{
    if (TANH) return tanhf(x);
    return fmaxf(x, 0.2f * x);  // LeakyReLU(0.2): the larger of x and 0.2 x (same values, two instructions)
}

// One 128-row tile through stage ST's three layers.  in[K0]: this thread's gathered input row (zeros beyond IN and
// for rows past the end of the list); out[OUT]: its output row.  wb: the stage's blob in shared memory.
template <int ST, int COLS = 128>
__device__ __forceinline__ void mlp_tile(Wg &g, const uint32_t *wb, const float *in, float *out)
{
    using S = Spec<ST>;
    using L = Blob<ST>;
    static_assert(COLS == 128 || S::OUT > 1, "the score heads need the 128-column map");
    const float *bias = reinterpret_cast<const float *>(wb + L::BIAS);
    store_a_row<S::K0, COLS>(g, in);
    if constexpr (S::OUT > 1) {
        {
            float v[S::H1];
            if constexpr (COLS == 64 && 3 * S::K0 / 2 + S::H1 > 64) {
                // (DagEncoder, K0 32: A takes 48 of the 64 columns, so layer 1 runs 16 output columns at a time)
                run_layer<S::K0, 16, S::H1, COLS>(g, wb + L::W1, 0);
                tc::tmem_ld_row<16>(g.trow + COL_D, v);
                run_layer<S::K0, 16, S::H1, COLS>(g, wb + L::W1, 16);
                tc::tmem_ld_row<16>(g.trow + COL_D, v + 16);
            } else {
                run_layer<S::K0, S::H1, S::H1, COLS>(g, wb + L::W1, 0);
                tc::tmem_ld_row<S::H1>(g.trow + COL_D, v);
            }
#pragma unroll
            for (int i = 0; i < S::H1; i++) v[i] = act<S::TANH>(v[i] + bias[i]);
            store_a_row<S::H1, COLS>(g, v);
        }
        run_layer<S::H1, S::H2, S::H2, COLS>(g, wb + L::W2, 0);
        {
            float v[S::H2];
            tc::tmem_ld_row<S::H2>(g.trow + COL_D, v);
#pragma unroll
            for (int i = 0; i < S::H2; i++) v[i] = act<S::TANH>(v[i] + bias[S::H1 + i]);
            store_a_row<S::H2, COLS>(g, v);
        }
        run_layer<S::H2, S::OUT, S::OUT, COLS>(g, wb + L::W3, 0);
        tc::tmem_ld_row<S::OUT>(g.trow + COL_D, out);
#pragma unroll
        for (int i = 0; i < S::OUT; i++) out[i] += bias[S::H1 + S::H2 + i];
    } else {
        // the score heads: 64-wide hidden layers computed 32 output columns at a time (D has 32 columns), the
        // final 64 -> 1 layer as a dot product in the row's thread
        float v[64];
        run_layer<S::K0, 32, S::H1>(g, wb + L::W1, 0);
        tc::tmem_ld_row<32>(g.trow + COL_D, v);
        run_layer<S::K0, 32, S::H1>(g, wb + L::W1, 32);   // (its barrier orders every thread's D read before the MMA)
        tc::tmem_ld_row<32>(g.trow + COL_D, v + 32);
#pragma unroll
        for (int i = 0; i < 64; i++) v[i] = act<S::TANH>(v[i] + bias[i]);
        store_a_row<64>(g, v);
        run_layer<64, 32, S::H2>(g, wb + L::W2, 0);
        tc::tmem_ld_row<32>(g.trow + COL_D, v);
        run_layer<64, 32, S::H2>(g, wb + L::W2, 32);
        tc::tmem_ld_row<32>(g.trow + COL_D, v + 32);
        const float *w3 = reinterpret_cast<const float *>(wb + L::W3V);
        float s = bias[S::H1 + S::H2];
#pragma unroll
        for (int i = 0; i < 64; i++) s = fmaf(w3[i], act<S::TANH>(v[i] + bias[S::H1 + i]), s);
        out[0] = s;
    }
    tc_fence_before();  // this tile's TMEM reads are ordered before the next tile's first MMA
}

// ------------------------------------------------------------------ building block / test hook
// out[n][max(OUT, 1)] = MLP_ST(x[n][IN]) for caller-provided rows (ssb_decima_mlp_rows)
template <int ST>
__global__ void __launch_bounds__(128) k_mlp_rows(const uint32_t *blob_all, const float *x, int n_rows, float *out)
{
    using S = Spec<ST>;
    using L = Blob<ST>;
    extern __shared__ __align__(128) uint32_t fsm[];
    __shared__ __align__(8) unsigned long long mbar_s;
    __shared__ uint32_t slot_s;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < L::WORDS / 4; i += 128)
        reinterpret_cast<uint4 *>(fsm)[i] = reinterpret_cast<const uint4 *>(blob_all + blob3_offset(ST))[i];
    if (warp == 0) tmem_alloc(smem_u32(&slot_s), COLS_PER_WG);
    if (tid == 0) mbar_init(smem_u32(&mbar_s), 1);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    Wg g;
    g.tmem = slot_s;
    g.trow = g.tmem + ((uint32_t)(warp * 32) << 16);
    g.mbar = smem_u32(&mbar_s);
    g.parity = 0; g.tid = tid; g.bar = 1;
    const int n_tiles = (n_rows + 127) >> 7;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row = tile * 128 + tid;
        float in[S::K0], o[S::OUT > 1 ? S::OUT : 1];
#pragma unroll
        for (int k = 0; k < S::K0; k++) in[k] = (row < n_rows && k < S::IN) ? x[(size_t)row * S::IN + k] : 0.0f;
        mlp_tile<ST>(g, fsm, in, o);
        if (row < n_rows) {
#pragma unroll
            for (int i = 0; i < (S::OUT > 1 ? S::OUT : 1); i++) out[(size_t)row * (S::OUT > 1 ? S::OUT : 1) + i] = o[i];
        }
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(g.tmem, COLS_PER_WG);
}

// ------------------------------------------------------------------ list-driven tile kernel
// One MLP over a row list built by the planning kernels (ssb_decima_tc.cuh: all nodes, sinks, the senders / receivers
// of one level, jobs, schedulable stages, executor-count rows): the launch sequence of round 1 with the tile routine
// above.  128 threads = one warpgroup per CTA, 128 TMEM columns, four CTAs per SM.
#ifndef SSB_TILE3_GATHER_CTAS
#define SSB_TILE3_GATHER_CTAS 5
#endif
#ifndef SSB_RCV_DEPTH
#define SSB_RCV_DEPTH 3
#endif
#ifndef SSB_TILE3_CTAS
#define SSB_TILE3_CTAS 8
#endif
namespace fused {
template <int ST> __device__ __forceinline__ void gather(const Params &p, int id, int level, float *in);
}
// resident CTAs per SM a stage's kernel is compiled for: eight 64-column TMEM contexts for the GNN MLPs, except the two
// gather-heavy stages (receivers: children's messages, jobs: the job's node rows; four 16-float rows in flight), which
// spill ~290 B per thread at the 64-register cap of eight -- six (85 registers) keeps them in registers; four 128-column
// contexts for the score heads
template <int ST> constexpr int tile3_ctas() { return Spec<ST>::OUT > 1 ? ((ST == tc::ST_RCV || ST == tc::ST_GLOB) ? SSB_TILE3_GATHER_CTAS : SSB_TILE3_CTAS) : 4; }
template <int ST>
__global__ void __launch_bounds__(128, tile3_ctas<ST>()) k_tile3(Params p, tc::TileArgs a)
{
    using S = Spec<ST>;
    using L = Blob<ST>;
    constexpr int COLS = S::OUT > 1 ? 64 : 128;  // the GNN MLPs fit the 64-column map: eight CTAs per SM
    const int n_rows = *a.count;
    if (n_rows <= 0) return;
    const int32_t *list = a.list + (a.offset ? *a.offset : 0);
    const int n_tiles = (n_rows + 127) >> 7;
    if ((int)blockIdx.x >= n_tiles) return;
    extern __shared__ __align__(128) uint32_t tsm[];
    __shared__ __align__(8) unsigned long long mbar_s;
    __shared__ uint32_t slot_s;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < L::WORDS / 4; i += 128)
        reinterpret_cast<uint4 *>(tsm)[i] = reinterpret_cast<const uint4 *>(p.pol_wblob3 + blob3_offset(ST))[i];
    if (warp == 0) tmem_alloc(smem_u32(&slot_s), COLS);
    if (tid == 0) mbar_init(smem_u32(&mbar_s), 1);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    Wg g;
    g.tmem = slot_s;
    g.trow = g.tmem + ((uint32_t)(warp * 32) << 16);
    g.mbar = smem_u32(&mbar_s);
    g.parity = 0; g.tid = tid; g.bar = 1;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row = tile * 128 + tid;
        int id = -1;
        if (row < n_rows) id = (ST == tc::ST_STAGE) ? row : list[row];
        float in[S::K0], o[S::OUT > 1 ? S::OUT : 1];
        if constexpr (ST == tc::ST_STAGE) {
            // id = position in the candidate list (pl_cand: node, pl_cand_job: job row, pl_cand_out: score slot)
#pragma unroll
            for (int i = 0; i < S::K0; i++) in[i] = 0.0f;
            if (id >= 0) {
                const int node = p.pl_cand[id], jid = p.pl_cand_job[id], b = node / p.Sc;
#pragma unroll
                for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)node * 5 + i];
                ld16(p.pol_h + (size_t)node * 16, *reinterpret_cast<float(*)[16]>(in + 5));
                ld16(p.pol_h_dag + (size_t)jid * 16, *reinterpret_cast<float(*)[16]>(in + 21));
                ld16(p.pol_h_glob + (size_t)b * 16, *reinterpret_cast<float(*)[16]>(in + 37));
            }
        } else {
            fused::gather<ST>(p, id, a.level, in);
            if constexpr (ST == tc::ST_MSG || ST == tc::ST_RCV) {
                const int pos = (a.offset ? *a.offset : 0) + row;
                if (a.x_save && id >= 0 && pos < a.x_cap) st16(a.x_save + (size_t)pos * 16, *reinterpret_cast<float(*)[16]>(in));
            }
        }
        mlp_tile<ST, COLS>(g, tsm, in, o);
        tc::scatter_row<ST>(p, id, o);
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(g.tmem, COLS);
}

// ====================================================================== the whole policy in ONE kernel
// DecimaScheduler.schedule (schedulers/decima/scheduler.py:71-99) for all environments: a persistent CTA (two
// warpgroups = two tile contexts, 256 TMEM columns) takes GROUPS of consecutive environments from a global cursor and
// runs the complete decision for its group -- observation adapter, level planning, mlp_prep, sinks, the
// message-passing levels (deepest first, parents OVERWRITE their embedding, :214-232), DagEncoder, GlobalEncoder,
// stage scores, sampling, executor-count scores, sampling -- with CTA-local barriers between the phases.  Within a
// phase the rows of ALL the group's environments are compacted into one list (shared memory), so a level that offers
// ~50 rows per environment still fills 128-row tiles.  Round 1 ran the same phases as ~50 dependent launches over all
// environments (one CUDA graph per decision); here the dependency chain is per group, the weights stay in shared
// memory and the activations in TMEM.
namespace fused {

constexpr int THREADS = 256, WARPS = 8, GMAX = 16, SPAN = 2048;

struct Args {
    const int32_t *forced_stage, *forced_num_exec;  // DEVICE i32[B] or nullptr (replayed / stored actions)
    int32_t *stage_idx_out, *num_exec_out;          // DEVICE i32[B] or nullptr (env-format action)
    int32_t *cursor;                                // DEVICE, zeroed before the launch: next group
    int run_adapter, advance_draws, group;          // group = environments per group (<= GMAX)
    const uint32_t *streams;                        // DEVICE u32[B]: each env's policy sampling stream
};

struct EnvInfo { int b, N, M, Ja, depth, node0, job0, ncand, cap, job_idx; };

struct Smem {
    // GNN weight blobs, resident for the whole kernel; the score heads share one buffer (loaded per group)
    static constexpr int PREP = 0;
    static constexpr int UPD = PREP + Blob<tc::ST_PREP>::WORDS;
    static constexpr int MSG = UPD + Blob<tc::ST_RCV>::WORDS;
    static constexpr int DAG = MSG + Blob<tc::ST_MSG>::WORDS;
    static constexpr int GLOB = DAG + Blob<tc::ST_DAG>::WORDS;
    static constexpr int HEAD = GLOB + Blob<tc::ST_GLOB>::WORDS;
    static constexpr int HEAD_WORDS = Blob<tc::ST_STAGE>::WORDS > Blob<tc::ST_EXEC>::WORDS ? Blob<tc::ST_STAGE>::WORDS
                                                                                           : Blob<tc::ST_EXEC>::WORDS;
    static constexpr int LIST = HEAD + HEAD_WORDS;            // u32[SPAN] row ids of the current phase
    static constexpr int SK = LIST + SPAN;                    // u64[WARPS][64] adapter scratch
    static constexpr int INFO = SK + WARPS * 64 * 2;          // EnvInfo[GMAX]
    static constexpr int CTL = INFO + GMAX * (int)(sizeof(EnvInfo) / 4);  // mbarriers, TMEM slot, counters
    static constexpr int WORDS = CTL + 16;
    static constexpr size_t BYTES = (size_t)WORDS * 4 + 128;
};

template <int ST> __device__ __forceinline__ int blob_at()
{
    return ST == tc::ST_PREP ? Smem::PREP : (ST == tc::ST_SINK || ST == tc::ST_RCV) ? Smem::UPD : ST == tc::ST_MSG ? Smem::MSG
         : ST == tc::ST_DAG ? Smem::DAG : ST == tc::ST_GLOB ? Smem::GLOB : Smem::HEAD;
}

__device__ __forceinline__ int job_of(const int32_t *dag_ptr, int Ja, int n)
{
    int lo = 0, hi = Ja;  // last j with dag_ptr[j] <= n
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (dag_ptr[mid] <= n) lo = mid; else hi = mid; }
    return lo;
}

// this thread's input row of stage ST.  id: PREP/SINK/MSG/RCV/DAG/STAGE flat node id (b * Sc + n), GLOB flat job id
// (b * Jc + j), EXEC b * Epad + c (c = candidate executor count - 1); -1: no row
template <int ST>
__device__ __forceinline__ void gather(const Params &p, int id, int level, float *in)
{
    using S = Spec<ST>;
#pragma unroll
    for (int i = 0; i < S::K0; i++) in[i] = 0.0f;
    if (id < 0) return;
    if constexpr (ST == tc::ST_PREP) {
#pragma unroll
        for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)id * 5 + i];
    } else if constexpr (ST == tc::ST_SINK) {
        ld16(p.pol_h_init + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in));
    } else if constexpr (ST == tc::ST_MSG) {
        ld16(p.pol_h + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in));
    } else if constexpr (ST == tc::ST_RCV) {
        // agg[u] = sum of the messages of u's children over the edges masked at this level, in edge order
        const int b = id / p.Sc, u = id - b * p.Sc;
        const int32_t *edges = p.obs_edges + (size_t)b * p.Mc * 2;
        const uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
        const int M = p.obs_hdr[b].num_edges;
        constexpr int RD = SSB_RCV_DEPTH;  // edges / message rows in flight
        for (int e0 = p.pol_row_start[id]; e0 < M; e0 += RD) {  // (a parent's edges are contiguous; RD in flight: 3 with 96 registers measured best)
            int2 uv[RD];
            uint64_t bits[RD];
#pragma unroll
            for (int q = 0; q < RD; q++) {
                const int e = e0 + q < M ? e0 + q : M - 1;
                uv[q] = *reinterpret_cast<const int2 *>(edges + 2 * e);
                bits[q] = ebits[e];
            }
            bool use[RD], more = true;
#pragma unroll
            for (int q = 0; q < RD; q++) {
                more = more && e0 + q < M && uv[q].x == u;
                use[q] = more && ((bits[q] >> level) & 1);
            }
            float m[RD][16];
#pragma unroll
            for (int q = 0; q < RD; q++)
                if (use[q]) ld16(p.pol_msg + ((size_t)b * p.Sc + uv[q].y) * 16, m[q]);
#pragma unroll
            for (int q = 0; q < RD; q++)
                if (use[q]) {
#pragma unroll
                    for (int i = 0; i < 16; i++) in[i] += m[q][i];
                }
            if (!more) break;
        }
    } else if constexpr (ST == tc::ST_DAG) {
#pragma unroll
        for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)id * 5 + i];
        ld16(p.pol_h + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in + 5));
    } else if constexpr (ST == tc::ST_GLOB) {
        // h_dag[j] = sum over the job's nodes of their DagEncoder terms (kept in pol_msg), in node order
        const int b = id / p.Jc, j = id - b * p.Jc;
        const int32_t *dag_ptr = p.obs_dag_ptr + (size_t)b * (p.Jc + 1);
        const int n1 = dag_ptr[j + 1];
        for (int n0 = dag_ptr[j]; n0 < n1; n0 += 4) {
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
    } else if constexpr (ST == tc::ST_STAGE) {
        const int b = id / p.Sc, n = id - b * p.Sc;
        const int j = job_of(p.obs_dag_ptr + (size_t)b * (p.Jc + 1), p.obs_hdr[b].num_active_jobs, n);
#pragma unroll
        for (int i = 0; i < 5; i++) in[i] = p.dec_feat[(size_t)id * 5 + i];
        ld16(p.pol_h + (size_t)id * 16, *reinterpret_cast<float(*)[16]>(in + 5));
        ld16(p.pol_h_dag + ((size_t)b * p.Jc + j) * 16, *reinterpret_cast<float(*)[16]>(in + 21));
        ld16(p.pol_h_glob + (size_t)b * 16, *reinterpret_cast<float(*)[16]>(in + 37));
    } else if constexpr (ST == tc::ST_EXEC) {
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
__device__ __forceinline__ void scatter(const Params &p, int id, const float *out)
{
    if (id < 0) return;
    if constexpr (ST == tc::ST_STAGE) p.pol_stage_logits[(size_t)(id / p.Sc) * p.Sc + p.pol_cand_rank[id]] = out[0];
    else tc::scatter_row<ST>(p, id, out);
}

// the tiles of the current list, split over the CTA's two warpgroups
template <int ST>
__device__ __forceinline__ void run_tiles(const Params &p, Wg &g, const uint32_t *sm, int n_rows, int level, int wg)
{
    using S = Spec<ST>;
    const uint32_t *list = sm + Smem::LIST;
    const int n_tiles = (n_rows + 127) >> 7;
    for (int tile = wg; tile < n_tiles; tile += 2) {
        const int row = tile * 128 + g.tid;
        const int id = row < n_rows ? (int)list[row] : -1;
        float in[S::K0], out[S::OUT > 1 ? S::OUT : 1];
        gather<ST>(p, id, level, in);
        mlp_tile<ST>(g, sm + blob_at<ST>(), in, out);
        scatter<ST>(p, id, out);
    }
}

// One phase = one MLP over the rows of the group selected by `pred(item) -> id or -1`, items [0, n_items) scanned in
// spans of SPAN (the list buffer's size); ends with a CTA barrier.
template <int ST, typename Pred>
__device__ __forceinline__ void run_phase(const Params &p, Wg &g, uint32_t *sm, int n_items, int level, Pred pred)
{
    uint32_t *list = sm + Smem::LIST;
    int *cnt = reinterpret_cast<int *>(sm + Smem::CTL + 8);
    const int tid = threadIdx.x, lane = tid & 31, wg = tid >> 7;
    for (int base = 0; base < n_items; base += SPAN) {
        if (tid == 0) *cnt = 0;
        __syncthreads();
        const int hi = min(base + SPAN, n_items);
        for (int it = base + tid; it - lane < hi; it += THREADS) {  // (whole warps iterate together)
            const int id = it < hi ? pred(it) : -1;
            const unsigned m = __ballot_sync(FULL, id >= 0);
            int pos = 0;
            if (lane == 0 && m) pos = atomicAdd(cnt, __popc(m));
            pos = __shfl_sync(FULL, pos, 0);
            if (id >= 0) list[pos + __popc(m & ((1u << lane) - 1))] = (uint32_t)id;
        }
        __syncthreads();
        run_tiles<ST>(p, g, sm, *cnt, level, wg);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(THREADS, 2) k_decima_fused(Params p, Args a)
{
    extern __shared__ unsigned char fsm_raw[];
    uint32_t *sm = reinterpret_cast<uint32_t *>((reinterpret_cast<uintptr_t>(fsm_raw) + 127) & ~uintptr_t(127));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wg = tid >> 7;
    EnvInfo *info = reinterpret_cast<EnvInfo *>(sm + Smem::INFO);
    int *ctl = reinterpret_cast<int *>(sm + Smem::CTL);  // [0..3] two mbarriers, [4] TMEM slot, [5] group, [8] list count
    {   // resident weights: the five GNN blobs, as built by k_build_blob (SINK and RCV share mlp_update's)
        const uint32_t *src = p.pol_wblob3;
        auto copy = [&](int dst, int st, int words) {
            const uint4 *s4 = reinterpret_cast<const uint4 *>(src + blob3_offset(st));
            uint4 *d4 = reinterpret_cast<uint4 *>(sm + dst);
            for (int i = tid; i < words / 4; i += THREADS) d4[i] = s4[i];
        };
        copy(Smem::PREP, tc::ST_PREP, Blob<tc::ST_PREP>::WORDS);
        copy(Smem::UPD, tc::ST_RCV, Blob<tc::ST_RCV>::WORDS);
        copy(Smem::MSG, tc::ST_MSG, Blob<tc::ST_MSG>::WORDS);
        copy(Smem::DAG, tc::ST_DAG, Blob<tc::ST_DAG>::WORDS);
        copy(Smem::GLOB, tc::ST_GLOB, Blob<tc::ST_GLOB>::WORDS);
    }
    if (warp == 0) tmem_alloc(smem_u32(ctl + 4), 2 * COLS_PER_WG);
    if (tid == 0) { mbar_init(smem_u32(ctl), 1); mbar_init(smem_u32(ctl + 2), 1); }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    Wg g;
    g.tmem = *reinterpret_cast<volatile uint32_t *>(ctl + 4) + wg * COLS_PER_WG;
    g.trow = g.tmem + ((uint32_t)((warp & 3) * 32) << 16);
    g.mbar = smem_u32(ctl + 2 * wg);
    g.parity = 0; g.tid = tid & 127; g.bar = 1 + wg;
    const uint32_t tmem_base = g.tmem - wg * COLS_PER_WG;
    uint64_t *Sk = reinterpret_cast<uint64_t *>(sm + Smem::SK) + warp * 64;
    const int G = a.group;

    for (;;) {
        if (tid == 0) ctl[5] = atomicAdd(a.cursor, 1);
        __syncthreads();
        const int e0 = ctl[5] * G;
        if (e0 >= p.B) break;
        const int ne = min(G, p.B - e0);
        // ---- per environment (one warp each): observation adapter, level bit sets per node, candidate ranks
        for (int i = warp; i < ne; i += WARPS) {
            const int b = e0 + i;
            if (a.run_adapter) {
                Sim sim(p, b, lane);
                sim.decima_obs_w(Sk);
                __syncwarp();
            }
            const ssb_obs_hdr &oh = p.obs_hdr[b];
            const bool live = !(oh.terminated || oh.error) && (!p.pol_active || p.pol_active[b]);
            const int N = live ? oh.num_nodes : 0, M = live ? oh.num_edges : 0, Ja = live ? oh.num_active_jobs : 0;
            const int depth = live ? p.dec_depth[b] : 0;
            unsigned long long *bits = p.pl_bits + (size_t)b * p.Sc * 2;
            const int32_t *edges = p.obs_edges + (size_t)b * p.Mc * 2;
            const uint64_t *ebits = p.dec_edge_bits + (size_t)b * p.Mc;
            const uint8_t *smask = p.dec_stage_mask + (size_t)b * p.Sc;
            int ncand = 0;
            for (int n0 = 0; n0 < N; n0 += 32) {
                const int n = n0 + lane;
                if (n < N) { bits[2 * n] = 0ull; bits[2 * n + 1] = 0ull; }
                const bool c = n < N && smask[n];
                const unsigned m = __ballot_sync(FULL, c);
                if (c) p.pol_cand_rank[(size_t)b * p.Sc + n] = ncand + __popc(m & ((1u << lane) - 1));
                ncand += __popc(m);
            }
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
            if (lane == 0) {
                EnvInfo x;
                x.b = b; x.N = N; x.M = M; x.Ja = Ja; x.depth = depth; x.node0 = 0; x.job0 = 0; x.ncand = ncand;
                x.cap = 0; x.job_idx = -1;
                info[i] = x;
                p.pl_ncand[b] = ncand;
            }
        }
        __syncthreads();
        if (tid == 0) {
            int n = 0, j = 0, d = 0;
            for (int i = 0; i < ne; i++) { info[i].node0 = n; info[i].job0 = j; n += info[i].N; j += info[i].Ja; d = max(d, info[i].depth); }
            ctl[9] = n; ctl[10] = j; ctl[11] = d;
        }
        __syncthreads();
        const int NT = ctl[9], JT = ctl[10], dmax = ctl[11];
        // item -> flat node id (b * Sc + n) / flat job id (b * Jc + j)
        auto node_of = [&](int it) {
            int i = 0;
            while (i + 1 < ne && it >= info[i + 1].node0) i++;
            return info[i].b * p.Sc + (it - info[i].node0);
        };
        auto job_item = [&](int it) {
            int i = 0;
            while (i + 1 < ne && it >= info[i + 1].job0) i++;
            return info[i].b * p.Jc + (it - info[i].job0);
        };
        const unsigned long long *bits_all = p.pl_bits;
        // ---- NodeEncoder (:191-234)
        run_phase<tc::ST_PREP>(p, g, sm, NT, 0, node_of);
        run_phase<tc::ST_SINK>(p, g, sm, NT, 0, [&](int it) {
            const int id = node_of(it);
            return (p.dec_depth[id / p.Sc] > 0 && bits_all[2 * (size_t)id + 1] == 0ull) ? id : -1;
        });
        for (int k = dmax - 1; k >= 0; k--) {  // reversed(edge_masks)
            run_phase<tc::ST_MSG>(p, g, sm, NT, k, [&](int it) {
                const int id = node_of(it);
                return ((bits_all[2 * (size_t)id] >> k) & 1ull) ? id : -1;
            });
            run_phase<tc::ST_RCV>(p, g, sm, NT, k, [&](int it) {
                const int id = node_of(it);
                return ((bits_all[2 * (size_t)id + 1] >> k) & 1ull) ? id : -1;
            });
        }
        // ---- DagEncoder (:244-257) and GlobalEncoder (:260-276)
        run_phase<tc::ST_DAG>(p, g, sm, NT, 0, node_of);
        run_phase<tc::ST_GLOB>(p, g, sm, JT, 0, job_item);
        for (int i = warp; i < ne; i += WARPS) {  // h_glob = sum over the active jobs, in job order
            if (lane < 16) {
                const int b = info[i].b;
                float s = 0.0f;
                for (int j = 0; j < info[i].Ja; j++) s += p.pol_g[((size_t)b * p.Jc + j) * 16 + lane];
                p.pol_h_glob[(size_t)b * 16 + lane] = s;
            }
        }
        {   // stage head's weights into the head buffer
            const uint4 *s4 = reinterpret_cast<const uint4 *>(p.pol_wblob3 + blob3_offset(tc::ST_STAGE));
            uint4 *d4 = reinterpret_cast<uint4 *>(sm + Smem::HEAD);
            for (int i = tid; i < Blob<tc::ST_STAGE>::WORDS / 4; i += THREADS) d4[i] = s4[i];
            fence_async_smem();
        }
        __syncthreads();
        // ---- stage scores (:279-320) over the schedulable stages
        run_phase<tc::ST_STAGE>(p, g, sm, NT, 0, [&](int it) {
            const int id = node_of(it);
            return p.dec_stage_mask[id] ? id : -1;
        });
        {   // executor-count head's weights replace the stage head's (all its tiles are done: run_phase ends in a barrier)
            const uint4 *s4 = reinterpret_cast<const uint4 *>(p.pol_wblob3 + blob3_offset(tc::ST_EXEC));
            uint4 *d4 = reinterpret_cast<uint4 *>(sm + Smem::HEAD);
            for (int i = tid; i < Blob<tc::ST_EXEC>::WORDS / 4; i += THREADS) d4[i] = s4[i];
            fence_async_smem();
        }
        // ---- stage sampling (utils.sample, decima/utils.py:19-23), one warp per environment
        for (int i = warp; i < ne; i += WARPS) {
            const int b = info[i].b, N = info[i].N, Ja = info[i].Ja, n_cand = info[i].ncand;
            const EnvHdr &h = p.hdr[b];
            const uint4 rw = philox4x32_10(h.policy_draws, a.streams[b], 4u, 0u, (uint32_t)h.seed, (uint32_t)(h.seed >> 32));
            const float u1 = ((float)(rw.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
            float lgprob = 0.0f, h_stage = 0.0f;
            const int stage_idx = n_cand > 0 ? sample_w(p.pol_stage_logits + (size_t)b * p.Sc, n_cand,
                                                        a.forced_stage ? a.forced_stage[b] : -1, u1, lane, lgprob, &h_stage) : -1;
            int job_idx = -1, cap = 0;
            if (stage_idx >= 0 && stage_idx < n_cand) {
                const uint8_t *smask = p.dec_stage_mask + (size_t)b * p.Sc;
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
                job_idx = job_of(p.obs_dag_ptr + (size_t)b * (p.Jc + 1), Ja, node);
                cap = p.dec_caps[(size_t)b * p.Jc + job_idx];
            }
            if (lane == 0) {
                int32_t *act = p.pol_action + (size_t)b * 4;
                act[0] = stage_idx; act[1] = job_idx; act[2] = 0; act[3] = n_cand;
                p.pol_lgprob[b] = lgprob;
                p.pol_entropy[b] = h_stage;  // completed below
                info[i].cap = cap; info[i].job_idx = job_idx;
            }
        }
        __syncthreads();
        // ---- executor-count scores (:338-385): cap rows per environment
        run_phase<tc::ST_EXEC>(p, g, sm, ne * p.Epad, 0, [&](int it) {
            const int i = it / p.Epad, c = it - i * p.Epad;
            return c < info[i].cap ? info[i].b * p.Epad + c : -1;
        });
        // ---- executor-count sampling, outputs
        for (int i = warp; i < ne; i += WARPS) {
            const int b = info[i].b, cap = info[i].cap;
            EnvHdr &h = p.hdr[b];
            const uint32_t pd = h.policy_draws;
            const uint4 rw = philox4x32_10(pd, a.streams[b], 4u, 0u, (uint32_t)h.seed, (uint32_t)(h.seed >> 32));
            const float u2 = ((float)(rw.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
            float lgprob = p.pol_lgprob[b], h_exec = 0.0f;
            int num_exec = 0;
            if (cap > 0)
                num_exec = sample_w(p.pol_exec_logits + (size_t)b * p.Epad, cap, a.forced_num_exec ? a.forced_num_exec[b] : -1,
                                    u2, lane, lgprob, &h_exec);
            __syncwarp();
            if (lane == 0) {
                int32_t *act = p.pol_action + (size_t)b * 4;
                act[2] = num_exec;
                p.pol_lgprob[b] = lgprob;
                // evaluate_actions: (stage entropy + exec entropy) / log(num_executors * nodes in the observation)
                const int N = p.obs_hdr[b].num_nodes;
                p.pol_entropy[b] = N > 0 ? (p.pol_entropy[b] + h_exec) / logf((float)(p.E * N)) : 0.0f;
                if (a.advance_draws && (!p.pol_active || p.pol_active[b])) h.policy_draws = pd + 1;
                if (a.stage_idx_out) a.stage_idx_out[b] = act[0];
                if (a.num_exec_out) a.num_exec_out[b] = 1 + num_exec;
            }
        }
        __syncthreads();
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 2 * COLS_PER_WG);
}

}  // namespace fused
}  // namespace fz
}  // namespace ssb
