// The optimizer half of one graph-replayable training step (tsb_train_step): AdamUniform (utils/optimizer.py:37-89)
// with every per-step scalar read from a device-resident schedule row selected by a device-side step counter, so that
// a captured sequence of steps replays without the host.  The energy half is the unchanged fused launch
// (launch_energy_grad).  Both kernels are ordinary launches (no programmatic dependent launch): they start only once
// the energy kernel of the same step has completed, and the next step's energy kernel, which is launched with
// programmatic stream serialisation, reads x only after its griddepcontrol.wait, i.e. after the apply kernel.
#include <cuda_runtime.h>

#include "tsb_kernels.cuh"

namespace tsb {
namespace {

// v >= 0: the order-preserving uint compare of non-negative floats (as the block maxima of tsb_kernels.cu).
__device__ __forceinline__ void train_block_max_to(float v, float *dst) {
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __shared__ float s_m[32];
  if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    float m = (threadIdx.x < (blockDim.x + 31) / 32) ? s_m[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int *>(dst), __float_as_uint(m));
  }
  __syncthreads();
}

// Pass 1: g = m_k * grad_e (+ grad_ext), the moments of adam_uniform_moments_kernel and their two global maxima
// (work[0] = max sqrt(m2_hat), work[1] = max |m1_hat|); block 0 records the step's energies in history[k].
__global__ void train_moments_kernel(const float *__restrict__ grad_e, const float *__restrict__ grad_ext,
                                     float *__restrict__ g1, float *__restrict__ g2, int64_t count, float b1, float b2,
                                     float omb1, float omb2, const float *__restrict__ schedule,
                                     const float *__restrict__ energy, float *__restrict__ history,
                                     const int32_t *step, int32_t n_steps, float *work) {
  const int k = *step;
  if (k < 0 || k >= n_steps) {                              // past the schedule: touch nothing, raise the flag
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned int *>(work + kTrainWorkFlag), 1u);
    return;
  }
  const float *row = schedule + 5 * size_t(k);
  const float m = row[0], inv_bc1 = row[2], inv_bc2 = row[3];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    float *h = history + 4 * size_t(k);
    h[0] = m * energy[0]; h[1] = energy[1]; h[2] = energy[2]; h[3] = m;
  }
  float mx2 = 0.f, mx1 = 0.f;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < count; i += int64_t(gridDim.x) * blockDim.x) {
    const float g = grad_ext ? fmaf(m, grad_e[i], grad_ext[i]) : m * grad_e[i];
    const float m1 = b1 * g1[i] + omb1 * g;                 // optimizer.py:61, as adam_uniform_moments_kernel
    const float m2 = b2 * g2[i] + omb2 * (g * g);           // optimizer.py:62
    g1[i] = m1; g2[i] = m2;
    mx2 = fmaxf(mx2, sqrtf(m2 * inv_bc2));                  // optimizer.py:68,74
    mx1 = fmaxf(mx1, fabsf(m1 * inv_bc1));                  // optimizer.py:67,83
  }
  train_block_max_to(mx2, work);
  train_block_max_to(mx1, work + 1);
}

// Pass 2: p -= lr_k * clamp(m1_hat / (1e-8 + max sqrt(m2_hat)))   (optimizer.py:74-88, as adam_uniform_apply_kernel).
// The last CTA (ticket in work[2]) re-zeroes the maxima and the ticket and advances the step counter.
__global__ void train_apply_kernel(float *__restrict__ p, const float *__restrict__ g1, int64_t count,
                                   const float *__restrict__ schedule, int32_t *step, int32_t n_steps, float *work) {
  const int k = *step;
  if (k < 0 || k >= n_steps) return;
  const float *row = schedule + 5 * size_t(k);
  const float lr = row[1], inv_bc1 = row[2], grad_limit = row[4];
  const float denom = 1e-8f + __ldcg(work);
  float f = inv_bc1 / denom;
  if (grad_limit > 0.f) {
    const float s = __ldcg(work + 1) / denom;               // max |gr|
    if (s > grad_limit) f *= grad_limit / s;
  }
  f *= lr;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < count; i += int64_t(gridDim.x) * blockDim.x) p[i] -= f * g1[i];
  __syncthreads();                                          // every thread of this CTA has read *step
  if (threadIdx.x == 0) {
    unsigned int *ticket = reinterpret_cast<unsigned int *>(work + 2);
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) { work[0] = 0.f; work[1] = 0.f; *ticket = 0u; *step = k + 1; }
  }
}

}  // namespace

cudaError_t launch_train_adam(float *p, const float *grad_e, const float *grad_ext, float *g1, float *g2, int64_t count,
                              double b1, double b2, const float *schedule, const float *energy, float *history,
                              int32_t *step, int32_t n_steps, float *work, cudaStream_t st) {
  int64_t g = (count + 255) / 256;
  const int grid = int(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));   // as the AdamUniform launches
  train_moments_kernel<<<grid, 256, 0, st>>>(grad_e, grad_ext, g1, g2, count, float(b1), float(b2), float(1.0 - b1),
                                             float(1.0 - b2), schedule, energy, history, step, n_steps, work);
  train_apply_kernel<<<grid, 256, 0, st>>>(p, g1, count, schedule, step, n_steps, work);
  return cudaGetLastError();
}

}  // namespace tsb
