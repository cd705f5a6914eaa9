// ssb_decima.cuh -- pieces shared by the Decima policy kernels (ssb_decima_tc.cuh): the weight
// layouts, 16-float row loads/stores and the softmax sampler.
//
// DecimaScheduler.schedule (schedulers/decima/scheduler.py:71-99): DAG-GNN encoder (NodeEncoder
// :173-241, DagEncoder :244-257, GlobalEncoder :260-276), stage score network (:279-320),
// executor-count score network (:323-385) and utils.sample (decima/utils.py:19-23).
#pragma once
#include "ssb_sim.cuh"

namespace ssb {

// ABI layout (dw): the tensors of models/decima/model.pt in state_dict order, each [out][in] row-major
// (42 tensors, 20 802 floats).  Device layout (dd): per layer the TRANSPOSED weight [in][out] followed
// by the bias, every tensor padded to a multiple of 4 floats (ssb_set_decima_weights does the re-layout);
// fz::k_build_blob turns it into the per-stage bf16 three-term weight blobs the tensor-core kernels copy to shared memory.
namespace dw {
constexpr int mlp(int in, int h1, int h2, int out) { return h1 * in + h1 + h2 * h1 + h2 + out * h2 + out; }
constexpr int TOTAL = mlp(5, 32, 16, 16) + 2 * mlp(16, 32, 16, 16) + mlp(21, 32, 16, 16) + mlp(16, 32, 16, 16) +
                      mlp(53, 64, 64, 1) + mlp(36, 64, 64, 1);
static_assert(TOTAL == 20802, "Decima parameter count");
// offsets of the seven MLPs in the ABI vector (W1 [h1][in], b1, W2 [h2][h1], b2, W3 [out][h2], b3 each)
constexpr int PREP = 0;
constexpr int MSG = PREP + mlp(5, 32, 16, 16);
constexpr int UPD = MSG + mlp(16, 32, 16, 16);
constexpr int DAG = UPD + mlp(16, 32, 16, 16);
constexpr int GLOB = DAG + mlp(21, 32, 16, 16);
constexpr int STAGE = GLOB + mlp(16, 32, 16, 16);
constexpr int EXEC = STAGE + mlp(53, 64, 64, 1);
}  // namespace dw
namespace dd {
__host__ __device__ constexpr int pad4(int n) { return (n + 3) & ~3; }
__host__ __device__ constexpr int layer(int in, int out) { return pad4(in * out) + pad4(out); }
__host__ __device__ constexpr int mlp(int in, int h1, int h2, int out)
{
    return layer(in, h1) + layer(h1, h2) + layer(h2, out);
}
constexpr int PREP = 0;
constexpr int MSG = PREP + mlp(5, 32, 16, 16);
constexpr int UPD = MSG + mlp(16, 32, 16, 16);
constexpr int DAG = UPD + mlp(16, 32, 16, 16);
constexpr int GLOB = DAG + mlp(21, 32, 16, 16);
constexpr int STAGE = GLOB + mlp(16, 32, 16, 16);
constexpr int EXEC = STAGE + mlp(53, 64, 64, 1);
constexpr int TOTAL = EXEC + mlp(36, 64, 64, 1);
}  // namespace dd

__device__ __forceinline__ void ld16(const float *p, float (&v)[16])
{
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float4 q = reinterpret_cast<const float4 *>(p)[i];
        v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    }
}
__device__ __forceinline__ void st16(float *p, const float (&v)[16])
{
#pragma unroll
    for (int i = 0; i < 4; i++) reinterpret_cast<float4 *>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}

// softmax-sample (or take `forced` if >= 0) over logits[0..n) ; returns the index, adds log prob; *entropy (optional)
// receives -sum p log p with the probabilities clamped to [eps, 1 - eps] (utils.evaluate, decima/utils.py:26-42)
__device__ inline int sample_w(const float *logits, int n, int forced, float u, int lane, float &lgprob,
                               float *entropy = nullptr)
{
    float mx = -INFINITY;
    for (int i = lane; i < n; i += 32) mx = fmaxf(mx, logits[i]);
    for (int off = 16; off; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, off));
    float sum = 0.0f;
    for (int i = lane; i < n; i += 32) sum += expf(logits[i] - mx);
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
    int idx = forced;
    if (idx < 0) {  // inverse-CDF draw, sequential over the candidates (lane 0)
        idx = n - 1;
        if (lane == 0) {
            float acc = 0.0f, target = u * sum;
            for (int i = 0; i < n; i++) {
                acc += expf(logits[i] - mx);
                if (acc > target) { idx = i; break; }
            }
        }
        idx = __shfl_sync(FULL, idx, 0);
    }
    if (idx >= 0 && idx < n) lgprob += logf(expf(logits[idx] - mx) / sum);
    if (entropy) {
        const float eps = 1.1920929e-07f;  // torch.finfo(float32).eps (torch.distributions.utils.clamp_probs)
        float hsum = 0.0f;
        for (int i = lane; i < n; i += 32) {
            const float pr = fminf(fmaxf(expf(logits[i] - mx) / sum, eps), 1.0f - eps);
            hsum -= pr * logf(pr);
        }
        for (int off = 16; off; off >>= 1) hsum += __shfl_xor_sync(FULL, hsum, off);
        *entropy = hsum;
    }
    return idx;
}

}  // namespace ssb
