// Device-side parameter block shared by tsb_kernels.cu (kernels) and tsb_capi.cu (C ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "tsb_plan.h"

namespace tsb {

struct KParams {
  // plan (read-only, built once by tsb_create)
  const unsigned char *stream;  // per-warp byte streams (operator rows + tet blocks)
  const float4 *X4;             // rest positions, float4 per staged vertex (STAGED: component-major; GLOBAL: by vertex id)
  const int32_t *vlist;         // STAGED: global vertex id per staged vertex (used when a component is not contiguous)
  const uint16_t *pos16;        // STAGED: staging position per staged vertex (bank-aware placement)
  const int32_t *pos_gid;       // STAGED: global vertex id per staging position
  const SegHdr *segs;
  const int2 *cta_seg;          // per CTA: [first segment, one past last)
  const uint2 *wdesc;           // per (CTA, warp): (stream offset / 16, stream bytes)
  const ushort2 *wseg;          // per (segment, warp): (row blocks, tet blocks)
  const float4 *Bt;             // AMIPS: rest inverses per streamed tet ([cell][row][slot] float4), or nullptr
  const int32_t *wtc0;          // AMIPS: first tet cell of every (segment, warp)
  const int32_t *orphans;       // vertices without tets
  int32_t n_orphans;
  int32_t n_components;
  // per-handle scratch (self-resetting)
  unsigned int *done;           // [n_components] warps that have stored their rows of a component
  double *cta_energy;           // [4*grid] (smooth, barrier, amips, 0) partials per CTA; a NaN-payload sentinel = "not written yet"
  float4 *u4g, *x4g;            // GLOBAL mode: displacement / position per vertex (written by the pre-pass)
  // per launch
  const float *x;               // [3n]
  float *grad;                  // [3n] or nullptr (energy only)
  float *energy_out;            // [3]: total, smooth, barrier
  const float *gradH_dev;       // optional device scalar
  float c1, c2, c3, gradH;      // c3: AMIPS coefficient (0 = term off)
  int32_t order;                // 2 or 4
  int32_t energy4;              // energy_out has 4 entries (total, smooth, barrier, amips)
  int32_t n;                    // vertices
  int32_t vh;                   // STAGED: half-buffer capacity in vertices
  int32_t ring_bytes;           // per-warp ring size = slots * cells_per_chunk cells
  int32_t cells_per_chunk;      // cells per TMA bulk copy (= per ring slot)
  int32_t ring_slots;
  int32_t stage_bytes;          // STAGED: bytes of the staging area at the start of shared memory
#ifdef TSB_TRACE
  unsigned long long *trace;    // profiling build only: [grid][16] phase stamps
#endif
};

struct LaunchConfig {
  int nw;          // warps per CTA (8 or 16)
  int grid;        // persistent CTAs
  int smem_bytes;  // dynamic shared memory
  int global;      // GLOBAL mode
  int amips;       // launch the AMIPS-capable instantiation
};

// Dynamic shared memory the kernel needs for a configuration (ring_slots chunks of cells_per_chunk cells per warp).
int energy_ring_bytes(int ring_slots, int cells_per_chunk, bool global);
int energy_smem_bytes(int nw, int ring_slots, int cells_per_chunk, int area_verts, bool global);
constexpr unsigned long long kEnergySentinel = 0x7FF8F00DBAADC0DEull;   // initial value of cta_energy
// Max co-resident CTAs per SM for a configuration (0 if it does not fit); also opts in to the smem size.
cudaError_t energy_occupancy(int nw, int smem_bytes, bool global, bool amips, int *ctas_per_sm);
cudaError_t launch_energy_grad(const KParams &p, const LaunchConfig &lc, cudaStream_t stream);

cudaError_t launch_scale(const float *g, int64_t count, float gradH, const float *gradH_dev, float *out, cudaStream_t s);
cudaError_t launch_grad_limit(float *g, int64_t count, float thr, float s, float *work4, cudaStream_t st);
cudaError_t launch_adam_uniform(float *p, const float *grad, float *g1, float *g2, int64_t count, double lr,
                                double b1, double b2, int step, double grad_limit, float *work4, cudaStream_t st);

// tsb_train.cu: the AdamUniform half of tsb_train_step (schedule row (m, lr, 1/(1-b1^t), 1/(1-b2^t), grad_limit)
// selected by *step).  work: [0..1] the two maxima, [2] the ticket, [kTrainWorkFlag] set when *step >= n_steps.
constexpr int kTrainWorkFlag = 3;
cudaError_t launch_train_adam(float *p, const float *grad_e, const float *grad_ext, float *g1, float *g2, int64_t count,
                              double b1, double b2, const float *schedule, const float *energy, float *history,
                              int32_t *step, int32_t n_steps, float *work, cudaStream_t st);

}  // namespace tsb
