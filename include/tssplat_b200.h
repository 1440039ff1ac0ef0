/* tssplat_b200 -- C ABI of the B200-native geometry-energy hot path of TetSphere Splatting.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry point
 * names the reference interface it replaces (paths relative to the reference checkout,
 * gmh14/tssplat @ 0241e9e3).  The reference-side binding a maintainer would add is shown in
 * INTEGRATION.md; the in-repo Python binding is tssplat_b200/_capi.py (ctypes).
 *
 * All device pointers are CUDA device pointers on the handle's device.  `stream` is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Every function returns 0 on
 * success and a negative TSB_E_* code on failure; tsb_last_error() gives the message.
 * A handle is not re-entrant (it owns scratch buffers), exactly like the reference's TetSpheres
 * object (tssplat_ext/tet_spheres/tet_spheres.h:37).
 */
#ifndef TSSPLAT_B200_H_
#define TSSPLAT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSB_VERSION 2

enum {
  TSB_OK = 0,
  TSB_E_INVALID = -1,   /* bad argument (null pointer, order not in {2,4}, sizes <= 0, ...)      */
  TSB_E_MESH = -2,      /* bad mesh: index out of range, zero-volume rest tet, non-manifold face */
  TSB_E_CUDA = -3,      /* a CUDA runtime call failed                                            */
  TSB_E_NOMEM = -4
};

typedef struct tsb_handle_s *tsb_handle_t;

typedef struct {
  int32_t warps_per_cta;    /* 0 = library default (16, one persistent CTA per SM); 8 = two CTAs per SM */
  int32_t laplacian_scale;  /* 0 = unscaled tet-graph Laplacian (what the reference requests:
                               tet_spheres.cpp:148 passes (1, 0)); 1 = rows divided by #nbrs    */
  int32_t ring_slots;       /* per-warp TMA ring depth in chunks of 6 cells: 0 = default (2); 2..8   */
  int32_t force_global;     /* 1: gather u/x from global memory instead of staging components in
                               shared memory (the mode used for components too large to stage)   */
  int32_t tet_cost_x100;    /* load-balance weight of one tet vs one operator entry, x100 (0 = default) */
  int32_t enable_amips;     /* 1: also keep the per-tet rest inverses (48 B/tet) so that tsb_energy_grad_ex
                               may add the AMIPS term; 0 (default): c3 must be 0                    */
  int32_t reserved[2];
} tsb_options_t;

/* Energy terms of tsb_energy_grad_ex.  c3 weighs the AMIPS term that BASELINE.json's north_star names:
 *   sum over tets with det F > 0 of  tr(F^T F) / (3 det(F)^(2/3)) - 1     (conformal AMIPS, Fu et al. 2015)
 * THE REFERENCE HAS NO SUCH TERM (nothing under /root/reference computes it: SURVEY.md F1), so there is no
 * reference oracle for it: it is verified against two fp64 restatements, finite differences and its known
 * answers (0 at rest and under similarity maps), never "against the reference".  Default off. */
typedef struct {
  float c1, c2;
  int32_t order;            /* 2 or 4 */
  float c3;                 /* AMIPS coefficient; 0 = exactly tsb_energy_grad */
  int32_t reserved[4];
} tsb_terms_t;

typedef struct {
  int32_t n;                /* vertices                                                          */
  int32_t nele;             /* tets                                                              */
  int32_t n_components;     /* connected components (= tet-spheres)                              */
  int32_t grid;             /* persistent CTAs per launch                                        */
  int32_t warps_per_cta;
  int32_t ctas_per_sm;
  int32_t mode_global;      /* 0 = components staged in shared memory, 1 = global gathers        */
  int32_t smem_bytes;       /* dynamic shared memory per CTA                                     */
  int32_t ring_slots;
  int32_t n_segments;       /* (CTA, component) work pieces                                      */
  int32_t n_boundary_faces;
  int32_t max_component_vertices;
  int64_t nnz;              /* off-diagonal entries of M = G^T L^T L G (per coordinate)          */
  int64_t nnz_padded;       /* entries stored in the row blocks (incl. padding)                  */
  int64_t device_bytes;     /* bytes of device memory owned by the handle                        */
  int64_t stream_bytes;     /* bytes one launch reads+writes: plan streams + rest + x + grad     */
} tsb_info_t;

/* Replaces TetSpheres::TetSpheres(int nv, double*, int ntet, int*) + TetSpheres::init
 * (tssplat_ext/tet_spheres/tet_spheres.cpp:119-126,140-203) and the libpgo operator builders it
 * calls (:148-149): builds the rows of M = G^T L^T L G (fp64, rounded to fp32 like :43-45), the
 * per-tet 1/det(Dm), and the per-warp work streams on the host, and uploads them to `device`.  rest_xyz: host float32 [3n] REST positions; tets: host int32
 * [4*nele], 0-based.  opt may be NULL. */
int tsb_create(const float *rest_xyz, const int32_t *tets, int32_t n, int32_t nele,
               const tsb_options_t *opt, int device, tsb_handle_t *out);

/* Replaces TetSpheres::~TetSpheres (tet_spheres.cpp:128-138); frees everything (no leaks). */
void tsb_destroy(tsb_handle_t h);

/* Message of the last failure on this handle (h may be NULL: last tsb_create failure). */
const char *tsb_last_error(tsb_handle_t h);

int tsb_get_info(tsb_handle_t h, tsb_info_t *info);

/* THE HOT PATH.  Replaces tet_spheres_smooth_barrier + tet_spheres_smooth_barrier_backward
 * (tssplat_ext/tet_spheres/tet_spheres_cuda.cu:118-195 and :197-263: 5 cuSPARSE SpMVs, 2 kernels,
 * 3 cuBLAS calls and 3 host syncs) with ONE kernel launch and no host sync:
 *   energy_out[0] = c1 * 1/2 x^T G^T L^T L G x + c2 * sum_t max(-det F_t,0)^order
 *   energy_out[1] = 1/2 x^T G^T L^T L G x    energy_out[2] = sum_t max(-det F_t,0)^order
 *   grad_out      = gradH * d energy_out[0] / d x          ([n,3] fp32, fully overwritten)
 * x_dev: device float32 [3n], contiguous.  gradH_dev: optional device float (0-dim tensor's
 * data pointer); when non-NULL it multiplies gradH (so pass gradH = 1).  grad_out_dev may be NULL
 * (energy only: replaces the forward alone).  order must be 2 or 4 (the reference silently
 * returns zeros otherwise: cu:57-63).  One launch may be in flight per handle at a time (the handle
 * owns counters and scratch, like the reference's TetSpheres: tet_spheres.h:37); launches on one
 * stream are chained with programmatic dependent launch.  Results are bitwise repeatable when no tet
 * is inverted; inverted tets add their barrier gradient with red.global.add.f32 (order-dependent
 * rounding in the affected vertices only). */
int tsb_energy_grad(tsb_handle_t h, const float *x_dev, float c1, float c2, int32_t order,
                    float gradH, const float *gradH_dev, float *energy_out_dev,
                    float *grad_out_dev, void *stream);

/* tsb_energy_grad plus the optional AMIPS term.  energy_out_dev: device float32 [4] = total, smoothness,
 * barrier, AMIPS (unweighted sums; total = c1*smooth + c2*barrier + c3*amips).  With terms->c3 == 0 the launch
 * is the very kernel tsb_energy_grad runs.  c3 != 0 needs a handle created with enable_amips = 1; its gradient
 * is added with red.global.add.f32 for every tet (order-dependent rounding). */
int tsb_energy_grad_ex(tsb_handle_t h, const float *x_dev, const tsb_terms_t *terms, float gradH,
                       const float *gradH_dev, float *energy_out_dev, float *grad_out_dev, void *stream);

/* Same computation for callers whose vertex positions live in HOST memory (e.g. a CPU-side
 * optimiser): copies x_host -> device, runs the fused launch, copies energy[3] and grad back,
 * asynchronously; the outputs are valid once `stream` has been synchronised and the host buffers
 * must stay valid until then (pinned memory makes the copies truly asynchronous).  Calls
 * alternate between two internal streams (upload -> kernel -> download, each with its own staging buffers;
 * only the kernels are ordered across the two), so successive calls pipeline: call i+1's upload overlaps
 * call i's kernel and download.  Consequences: x_host must be fully
 * written by the CPU when the call is made (the upload is NOT ordered after earlier work queued on
 * `stream`), and the handle must not be used through tsb_energy_grad on another stream until `stream` has
 * been synchronised.  grad_out_host may be NULL.
 * Replaces the reference's implicit host round trips (the CPU scalar at tet_spheres_cuda.cu:194 and
 * the caller's .cpu() of the gradient). */
int tsb_energy_grad_host(tsb_handle_t h, const float *x_host, float c1, float c2, int32_t order,
                         float gradH, float *energy_out_host, float *grad_out_host, void *stream);

/* out = gradH * (*gradH_dev) * g  -- the cublasSscal at tet_spheres_cuda.cu:257-258 without the
 * .item() sync.  In-place allowed. */
int tsb_scale(const float *g_dev, int64_t count, float gradH, const float *gradH_dev,
              float *out_dev, void *stream);

/* Replaces tet_spheres_grad_limit (tet_spheres_cuda.cu:265-303) with what it was meant to do
 * (the reference reads grad[0] instead of the arg-max element and is unused by the trainer):
 * if max|grad| > s_threshold, grad *= s / max|grad|.  No host sync. */
/* work_dev: device float32 [4] scratch owned by the caller (zero-initialised once; the kernels leave
 * it zeroed), one per concurrently used stream -- like tsb_adam_uniform_step. */
int tsb_grad_limit(float *grad_dev, int64_t count, float s_threshold, float s, float *work_dev, void *stream);

/* "Next" row (f)1: AdamUniform.step (utils/optimizer.py:37-89) as two launches and no sync.
 * p, g1, g2: device float32 [count]; step is the 1-based step number AFTER increment.  lr and the
 * betas are doubles (Python floats) so that 1-beta and the bias corrections round as in the reference.
 * grad_limit <= 0 disables the clamp (optimizer.py:76-86).  work_dev: device float32 [4]
 * scratch owned by the caller (zero-initialised once; the kernels leave it zeroed). */
int tsb_adam_uniform_step(float *p_dev, const float *grad_dev, float *g1_dev, float *g2_dev,
                          int64_t count, double lr, double beta1, double beta2, int32_t step,
                          double grad_limit, float *work_dev, void *stream);

/* State of tsb_train_step.  All buffers are caller-owned device memory on the handle's device.  The schedule row of
 * step k (0-based, k = *step) holds what the reference's loop changes on every step (trainer.py:71-132,
 * energies/smooth_barrier.py:47-63, utils/optimizer.py:37-89), each computed in double on the host and rounded to
 * float: the coefficient multiplier m of coeff_scheduler, the learning rate, the two bias corrections
 * 1/(1-beta^(k+1)) and the grad_limit value (<= 0: no clamp). */
typedef struct {
  float *g1, *g2;            /* [3n] Adam moments (zero-initialised by the caller), as AdamUniform's state g1, g2      */
  float *grad;               /* [3n] scratch: the energy gradient of the fused launch                              */
  float *energy;             /* [4]  scratch: energy_out of the fused launch                                       */
  const float *schedule;     /* [n_steps][5]: m, lr, 1/(1-b1^t), 1/(1-b2^t), grad_limit                            */
  float *history;            /* [n_steps][4]: loss = m * energy[0], smoothness, barrier, m; row k written by step k */
  int32_t *step;             /* device counter: steps taken = schedule row of the next step (zero it to start)     */
  float *work;               /* [8] scratch, zero-initialised once.  [0..2] are left zeroed by every step; [3] != 0
                                records that a step ran with *step >= n_steps (it then left everything untouched)   */
  int32_t n_steps;
  double beta1, beta2;       /* Adam betas (1 - beta is formed in double, like the reference's Python)             */
} tsb_train_state_t;

/* One step of the reference's geometry loop: the fused energy + gradient launch with the base coefficients c1, c2
 * (gradH = 1) into st->grad / st->energy, then g = m * grad (+ grad_ext_dev, e.g. the image loss's gradient of the
 * vertex positions; may be NULL) and AdamUniform with the schedule row *step, which updates x_dev, g1, g2 in place,
 * writes history[*step] and increments *step -- three launches (four in global-gather mode), no host sync, no
 * host-side state that changes between calls.  coeff_scheduler scales c1 and c2 by the same m, so m multiplies the
 * gradient (and the energy in the history) instead of the coefficients.  The barrier order is an argument: it
 * changes once (smooth_barrier.py:61-63), so a caller records one sequence per order.
 * Replaces, per step: SmoothnessBarrierFunc forward + backward (energies/smooth_barrier.py:9-31,60-67),
 * coeff_scheduler (:47-58), AdamUniform.step (utils/optimizer.py:37-89) and the LR scheduler step
 * (trainer.py:57-58,128-133).
 * Safe to capture in a CUDA graph: every per-step value is read on the device.  Inside a graph x_dev, grad_ext_dev
 * and the state's pointers are the ones given at capture time (rewrite the buffers' contents, not the pointers).
 * One launch may be in flight per handle, as for tsb_energy_grad.  work holds a ticket: one state per concurrently
 * used stream. */
int tsb_train_step(tsb_handle_t h, float *x_dev, const float *grad_ext_dev, float c1, float c2, int32_t order,
                   const tsb_train_state_t *st, void *stream);

/* ---- "Next" row (f)2: surface gather + vertex-normal splat ------------------------------------------------
 * Replaces `tet_v[surface_vid]` (geometry/tetmesh_geometry.py:33) and `_compute_vertex_normal`
 * (geometry/tetmesh_geometry.py:39-66) and their autograd backward.  surface_vid: host int32 [nsv] tet-mesh
 * vertex of each surface vertex (unique); surface_f: host int32 [3*nsf] triangles over surface-vertex ids.
 * One handle may serve one stream at a time (it owns a backward scratch array). */
typedef struct tsb_surface_s *tsb_surface_t;
int tsb_surface_create(const int32_t *surface_vid, int32_t nsv, const int32_t *surface_f, int32_t nsf,
                       int32_t n_tet_vertices, int device, tsb_surface_t *out);
void tsb_surface_destroy(tsb_surface_t s);
const char *tsb_surface_last_error(tsb_surface_t s);
/* v_pos_dev / v_nrm_dev: device float32 [3*nsv]; either may be NULL.  Normals: sum of cross(v1-v0, v2-v0) over the
 * incident faces in fixed order, (0,0,1) where |n|^2 <= 1e-20, then n / max(|n|, 1e-12). */
int tsb_surface_forward(tsb_surface_t s, const float *tet_v_dev, float *v_pos_dev, float *v_nrm_dev, void *stream);
/* grad_tet_v_dev: device float32 [3*n_tet_vertices], fully overwritten (zero for non-surface vertices);
 * grad_v_pos_dev / grad_v_nrm_dev: upstream gradients [3*nsv], either may be NULL. */
int tsb_surface_backward(tsb_surface_t s, const float *tet_v_dev, const float *grad_v_pos_dev,
                         const float *grad_v_nrm_dev, float *grad_tet_v_dev, void *stream);

/* ---- "Next" row (f)3: surface extraction on the GPU --------------------------------------------------------
 * Replaces get_surface_vf (geometry/mesh_utils.py:5-35; re-run by reset() / permute_surface_v(),
 * geometry/tetmesh_geometry.py:164-170,369-371) with identical output: the faces that belong to exactly one tet, in
 * lexicographic order of their sorted vertex triple, each in the orientation its tet gives it (face k opposite local
 * vertex k: (1,2,3), (0,3,2), (0,1,3), (0,2,1)), re-indexed into the increasing list of surface vertex ids.
 * tets_host: host int32 [4*nele], 0-based, entries in [0, n).  On success *surface_vid_out (int32 [*nsv_out]) and
 * *surface_f_out (int32 [3 * *nsf_out]) are host arrays owned by the caller: release them with tsb_free_host.
 * Synchronous (a setup call); errors are reported through tsb_setup_last_error (thread-local). */
int tsb_surface_extract(const int32_t *tets_host, int32_t nele, int32_t n, int device, int32_t *nsv_out,
                        int32_t *nsf_out, int32_t **surface_vid_out, int32_t **surface_f_out);
void tsb_free_host(void *p);
const char *tsb_setup_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* TSSPLAT_B200_H_ */
