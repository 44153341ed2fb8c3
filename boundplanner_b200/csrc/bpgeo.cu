// bpgeo.cu -- sm_100a kernels and the C ABI of libbpgeo.so (see include/bpgeo.h).
//
// Kernel map (reference sites in the per-kernel comments):
//   k_closest_points        K1  compute_set_projs          ConvexSetFinder.py:465-489
//   k_closest_points_line   K2  compute_set_projs_line     ConvexSetFinder.py:491-510
//   k_poly_point            K3  compute_polyhedron         ConvexSetFinder.py:423-463
//   k_poly_line             K3' greedy loop of find_set_collision_avoidance :309-375
//   k_mvie                  K4  mvie_socp / mvie_socp_fixed_mid  :512-562
//   (k_poly_point, k_mvie) x max_iter + k_mvie(final) = K5 find_set_around_point :190-240
//   k_pair_feasible         K6  set_intersection           BoundPlanner.py:774-798
//   k_fk                    K7  RobotModel.fk_pos/_col/hom_transform/jacobian :146-231
//
// Layout in HBM: the scene is six SoA columns (lbx,lby,lbz,ubx,uby,ubz) of N
// doubles, already inflated; a convex set is m rows (a0,a1,a2 | b) in
// A[S,m_max,3], b[S,m_max]; per-seed loop state lives in a SeedState array in
// the caller-provided workspace.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/bpgeo.h"
#include "bp_math.cuh"
#include "bp_mvie.cuh"
#include "bp_mvie_warp.cuh"
#include "bp_mvie_fixed_r.cuh"
#include "bp_lp.cuh"
#include "bp_lp_warp.cuh"
#include "bp_fk.cuh"

// ---------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int bp_fail(const char* what, cudaError_t e = cudaSuccess) {
  if (e != cudaSuccess)
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  else
    snprintf(g_err, sizeof(g_err), "%s", what);
  return 1;
}
#define BP_CUDA(call)                                   \
  do {                                                  \
    cudaError_t e_ = (call);                            \
    if (e_ != cudaSuccess) return bp_fail(#call, e_);   \
  } while (0)

struct bp_scene {
  double* cols;   // device, 6 * cap doubles: lbx | lby | lbz | ubx | uby | ubz (stride cap)
  int n;          // obstacles of a single scene, or of the largest scene of a batch
  int cap;
  double inflate;
  int* seg_off;   // device [n_seg + 1] or NULL: a batch of scenes stored back to back (one per planning query)
  int n_seg;
  // general polytope obstacles (bp_scene_create_polytopes): cols then hold the obstacles' bounding boxes
  double* rows;   // device [n, BP_OBS_ROWS, 4] (a0,a1,a2,b), zero rows (b = 10) after the last real one, or NULL
  int* nrows;     // device [n]
  double* verts;  // device [n, vmax, 3]
  int* nverts;    // device [n]
  int vmax;
  // scene batches: host copy of seg_off (bp_plan_run checks its inputs against it without a device round trip)
  int* seg_off_host;
  // capacities of rows / nrows / nverts (obstacles) and verts (doubles) of a polytope scene
  int pcap;
  size_t vcap;
  // staging of the batch updates (bp_scene_update_batch, bp_scene_update_polytopes_batch): pinned host and device
  void* stage_h;
  void* stage_d;
  size_t stage_h_cap, stage_d_cap;
};

struct SceneView {
  const double* lb[3];
  const double* ub[3];
  int n;
  const double* rows;     // polytope scene (else NULL): see bp_scene
  const int* nrows;
  const double* verts;
  const int* nverts;
  int vmax;
  const int* seg_off;     // scene batch: obstacle range of scene k is [seg_off[k], seg_off[k+1])
  const int* item_seg;    // scene index of every seed / segment (device, [S]) when seg_off != NULL
  int staged;             // lb / ub point into shared memory (stage_scene)
};

static SceneView view_of(const bp_scene* s) {
  SceneView v;
  for (int k = 0; k < 3; ++k) {
    v.lb[k] = s->cols + (size_t)k * s->cap;
    v.ub[k] = s->cols + (size_t)(3 + k) * s->cap;
  }
  v.n = s->n;
  v.rows = s->rows; v.nrows = s->nrows; v.verts = s->verts; v.nverts = s->nverts; v.vmax = s->vmax;
  v.seg_off = s->seg_off;
  v.item_seg = nullptr;
  v.staged = 0;
  return v;
}

static SceneView view_of(const bp_scene* s, const int* item_seg) {
  SceneView v = view_of(s);
  v.item_seg = item_seg;
  return v;
}

// the scene seen by work item `item`: the whole table, or the item's segment of a scene batch
__device__ __forceinline__ SceneView scene_of_item(const SceneView& sc, int item) {
  if (!sc.seg_off || !sc.item_seg) return sc;
  const int k = sc.item_seg[item];
  const int o = sc.seg_off[k];
  SceneView v;
#pragma unroll
  for (int a = 0; a < 3; ++a) { v.lb[a] = sc.lb[a] + o; v.ub[a] = sc.ub[a] + o; }
  v.n = sc.seg_off[k + 1] - o;
  // polytope batches: the obstacles' rows / vertex lists are stored back to back like the bounding boxes
  v.rows = sc.rows ? sc.rows + (size_t)o * BP_OBS_ROWS * 4 : nullptr;
  v.nrows = sc.rows ? sc.nrows + o : nullptr;
  v.verts = sc.rows ? sc.verts + (size_t)o * sc.vmax * 3 : nullptr;
  v.nverts = sc.rows ? sc.nverts + o : nullptr;
  v.vmax = sc.vmax;
  v.seg_off = nullptr;
  v.item_seg = nullptr;
  v.staged = 0;
  return v;
}

// Per-seed state of the IRIS loop (find_set_around_point, :190-240)
struct SeedState {
  double Q[9];      // q_ellipse
  double p[3];      // p_seed (moves when the centre is free)
  double det, det_old;
  int k;            // loop counter
  int active;       // still inside the while loop
  int status;
  int rows_peak;    // largest row count any pass handed to the MVIE (the reference raises above 20, quirk Q5)
};

struct Vec3 { double v[3]; };

#ifdef BPGEO_PROFILE
// profile build only (tools/prof_phases.py): per-seed cycle counters of the fused loop
__device__ long long g_prof[4 * 65536];   // [seed][poly cycles, mvie cycles, passes, total]
__device__ long long g_prof_pair[128];        // [0..63] histogram of Newton iterations per LP (bucket = iters / 2), [64] LPs, [65] sum of iterations, [66] max warp cycles, [67] answers 1
__device__ long long g_prof_poly[8 * 65536];   // [cta][phase1, argmin, refine, halfspace, delete scan, picks, refine rounds, qps of thread 0]
// (accumulated in registers and written once per pass: a global read-modify-write per lap costs ~600 cycles)
#define BP_PPROF_MARK() long long pprof_t_ = clock64(); long long pprof_a_[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define BP_PPROF_LAP(slot) { const long long now_ = clock64(); pprof_a_[slot] += now_ - pprof_t_; pprof_t_ = now_; }
#define BP_PPROF_COUNT(slot) { pprof_a_[slot] += 1; }
#define BP_PPROF_ADDN(slot, n) { pprof_a_[slot] += (n); }
#define BP_PPROF_FLUSH() { if (threadIdx.x == 0 && blockIdx.x < 65536) { for (int q_ = 0; q_ < 8; ++q_) g_prof_poly[8 * blockIdx.x + q_] += pprof_a_[q_]; } }
#define BP_PROF_T0() const long long prof_t0_ = clock64()
#define BP_PROF_ADD(slot) if ((threadIdx.x & 31) == 0 && blockIdx.x < 65536) g_prof[4 * blockIdx.x + (slot)] += clock64() - prof_t0_
#else
#define BP_PROF_T0()
#define BP_PROF_ADD(slot)
#define BP_PPROF_MARK()
#define BP_PPROF_LAP(slot)
#define BP_PPROF_COUNT(slot)
#define BP_PPROF_ADDN(slot, n)
#define BP_PPROF_FLUSH()
#endif


// ---------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}

__device__ __forceinline__ void tma_store_1d(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void load_box(const SceneView& sc, int j, double* lb, double* ub) {
  if (sc.staged) {                      // columns staged in shared memory (stage_scene): plain loads
#pragma unroll
    for (int k = 0; k < 3; ++k) { lb[k] = sc.lb[k][j]; ub[k] = sc.ub[k][j]; }
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lb[k] = __ldg(sc.lb[k] + j);
      ub[k] = __ldg(sc.ub[k] + j);
    }
  }
}

// Stage the six scene columns of this CTA's scene in shared memory with TMA bulk copies (cp.async.bulk, one
// elected thread, mbarrier completion): every later box read of the polyhedron passes (bounds, sweeps, exact
// QPs: ~4 N reads per pass) is then a shared-memory load instead of an L1/L2 access.  dst: 6 * ncap doubles,
// ncap = n rounded up to even (16-byte bulk granularity).  All threads call it; returns the staged view.
__device__ __forceinline__ SceneView stage_scene(const SceneView& sc, double* dst, uint64_t* bar) {
  const int ncap = (sc.n + 1) & ~1;
  const uint32_t bytes = (uint32_t)ncap * 8u;
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(6u * bytes) : "memory");
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       smem_u32(dst + (size_t)k * ncap)), "l"(sc.lb[k]), "r"(bytes), "r"(smem_u32(bar)) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       smem_u32(dst + (size_t)(3 + k) * ncap)), "l"(sc.ub[k]), "r"(bytes), "r"(smem_u32(bar)) : "memory");
    }
  }
  __syncthreads();                      // the barrier is initialised before anybody waits on it
  mbar_wait(bar, 0);
  SceneView v = sc;
#pragma unroll
  for (int k = 0; k < 3; ++k) { v.lb[k] = dst + (size_t)k * ncap; v.ub[k] = dst + (size_t)(3 + k) * ncap; }
  v.staged = 1;
  return v;
}

// (value, index) argmin across the block; ties -> smallest index (np.argmin, quirk Q11).
// Every thread returns the block result.  red_* are [2][32] ping-pong buffers.
__device__ __forceinline__ void block_argmin(double& val, int& idx, double (*red_val)[32], int (*red_idx)[32],
                                             int& buf) {
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    double ov = __shfl_xor_sync(full, val, off);
    int oi = __shfl_xor_sync(full, idx, off);
    if (ov < val || (ov == val && oi < idx)) { val = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) { red_val[buf][warp] = val; red_idx[buf][warp] = idx; }
  __syncthreads();
  double bv = red_val[buf][0];
  int bi = red_idx[buf][0];
  for (int w = 1; w < nw; ++w) {
    double ov = red_val[buf][w];
    int oi = red_idx[buf][w];
    if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  val = bv; idx = bi;
  buf ^= 1;
}

struct PassMetric {
  double Q[9];
  double G[9];       // Q Q^T (normals, :440)
  BpMetric mt;       // M = Q^T Q (QP objective == squared dist, :429)
};

__device__ __forceinline__ void pass_metric_init(const double* Q, PassMetric* pm) {
#pragma unroll
  for (int k = 0; k < 9; ++k) pm->Q[k] = Q[k];
  double M[9];
  bp_mat3_ata(Q, M);
  bp_mat3_mul_bt(Q, Q, pm->G);
  bp_metric_init(M, &pm->mt);
}

// closest point of box j to p in the pass metric; returns dist (:429)
__device__ __forceinline__ double closest_on_box(const PassMetric& pm, const double* p, const double* lb,
                                                 const double* ub, double* y) {
  double lo[3], hi[3], z[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { lo[k] = lb[k] - p[k]; hi[k] = ub[k] - p[k]; }
  int mask = bp_box_qp(pm.mt, lo, hi, z);
  bp_box_point(p, lb, ub, z, mask, y);
  double zz[3] = {y[0] - p[0], y[1] - p[1], y[2] - p[2]};
  double w[3];
  bp_mat3_vec(pm.Q, zz, w);
  return sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
}

struct GlobalRows4 {
  const double* r;
  __device__ __forceinline__ double a(int i, int k) const { return __ldg(r + 4 * i + k); }
  __device__ __forceinline__ double b(int i) const { return __ldg(r + 4 * i + 3); }
};

// ---------------------------------------------------------------------------
// K1 test hook / batched compute_set_projs
// ---------------------------------------------------------------------------
__global__ void k_closest_points(SceneView sc, const double* __restrict__ seeds, const double* __restrict__ q_inv,
                                 double* __restrict__ y_out, double* __restrict__ dist_out) {
  const int s = blockIdx.y;
  double E[9], Q[9], p[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) E[k] = q_inv[(size_t)s * 9 + k];
#pragma unroll
  for (int k = 0; k < 3; ++k) p[k] = seeds[(size_t)s * 3 + k];
  bp_inv3(E, Q);
  PassMetric pm;
  pass_metric_init(Q, &pm);
  BpPolyMetric pmq;
  if (sc.rows) {
    double M9[9];
    bp_mat3_ata(pm.Q, M9);
    bp_poly_metric_init(M9, &pmq);
  }
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < sc.n; j += gridDim.x * blockDim.x) {
    double lb[3], ub[3], y[3];
    double d;
    if (sc.rows) {                                 // general polytope: serial walk over the candidates
      GlobalRows4 rows{sc.rows + (size_t)j * BP_OBS_ROWS * 4};
      if (bp_polytope_qp(pmq, rows, sc.nrows[j], p, y)) {
        const double zz[3] = {y[0] - p[0], y[1] - p[1], y[2] - p[2]};
        double w[3];
        bp_mat3_vec(pm.Q, zz, w);
        d = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
      } else {
        y[0] = y[1] = y[2] = 0.0;
        d = BP_INF;
      }
    } else {
      load_box(sc, j, lb, ub);
      d = closest_on_box(pm, p, lb, ub, y);
    }
    size_t o = (size_t)s * sc.n + j;
    y_out[3 * o] = y[0]; y_out[3 * o + 1] = y[1]; y_out[3 * o + 2] = y[2];
    dist_out[o] = d;
  }
}

// ---------------------------------------------------------------------------
// K2 test hook / batched compute_set_projs_line
// ---------------------------------------------------------------------------
__global__ void k_closest_points_line(SceneView sc, const double* __restrict__ p0s, const double* __restrict__ p1s,
                                      double* __restrict__ x_out, double* __restrict__ phi_out) {
  const int s = blockIdx.y;
  double p0[3], d[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { p0[k] = p0s[(size_t)s * 3 + k]; d[k] = p1s[(size_t)s * 3 + k] - p0[k]; }
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < sc.n; j += gridDim.x * blockDim.x) {
    double lb[3], ub[3], x[3], d2;
    double phi;
    if (sc.rows) {                                 // general polytope: serial walk over the candidates
      GlobalRows4 rows{sc.rows + (size_t)j * BP_OBS_ROWS * 4};
      if (!bp_seg_polytope_qp(rows, sc.nrows[j], 0.001, p0, d, x, &phi, &d2)) { x[0] = x[1] = x[2] = 0.0; phi = -1.0; }
      size_t o = (size_t)s * sc.n + j;
      x_out[3 * o] = x[0]; x_out[3 * o + 1] = x[1]; x_out[3 * o + 2] = x[2];
      phi_out[o] = phi;
      continue;
    }
    load_box(sc, j, lb, ub);
#pragma unroll
    for (int k = 0; k < 3; ++k) { lb[k] += 0.001; ub[k] -= 0.001; }   // b - 0.001 (:496)
    phi = bp_seg_box(p0, d, lb, ub, x, &d2);
    size_t o = (size_t)s * sc.n + j;
    x_out[3 * o] = x[0]; x_out[3 * o + 1] = x[1]; x_out[3 * o + 2] = x[2];
    phi_out[o] = phi;
  }
}

// ---------------------------------------------------------------------------
// K3: one compute_polyhedron pass, one CTA per seed (ConvexSetFinder.py:423-463)
//   phase 1: every thread solves the box QP of its obstacles (j = tid + k*T)
//            and keeps dist[j] in shared memory (dead obstacles: +inf);
//   phase 2: greedy loop -- block argmin, halfspace from the winner (its QP is
//            re-solved redundantly by every thread instead of storing y[N,3]),
//            vertex test over the surviving obstacles.  One barrier per pick.
// mode 0: standalone pass (bp_polyhedron); mode 1: inside the IRIS loop (checks
// and updates the SeedState loop control, :203-207).
// ---------------------------------------------------------------------------
struct PolyParams {
  const double* seeds;       // [S,3]      (mode 0)
  const double* q_ellipse;   // [S,9]      (mode 0)
  const double* init_rows;   // [S,6,4]    (mode 0)
  SeedState* state;          // [S]        (mode 1)
  double ws_rows[6];         // b of the 6 workspace rows: ub0,-lb0,ub1,-lb1,ub2,-lb2 (mode 1)
  double* A;
  double* b;
  int* m;
  int* status;
  int m_max;
  int mode;
  int max_iter;
  int cache_y;               // closest points kept in shared memory (y[3][N] after dist[N])
  int shell;                 // box scene whose key table + shell fit in shared memory: poly_pass_shell
  int row_cap;               // > 0: stop a seed whose pass produced more rows (reference: 20, quirk Q5)
};

// (value, index) argmin of the lazy distance table: key = |entry| >= 0 (an exact distance or a lower bound of
// one), ties -> bounds before exact values (a bound that ties with the best exact distance must still be
// refined), then the smallest index (np.argmin, quirk Q11).  Non-negative doubles order like their bit patterns,
// so the warp stage is three integer redux.sync minima (high word, low word, code) instead of a 5-round shuffle
// butterfly.  With WITH_EX the smallest EXACT distance of the block is reduced the same way into `ex`.
__device__ __forceinline__ double warp_min_nonneg(double v) {
  const unsigned full = 0xffffffffu;
  const unsigned hi = (unsigned)__double2hiint(v);
  const unsigned mh = __reduce_min_sync(full, hi);
  const unsigned lo = hi == mh ? (unsigned)__double2loint(v) : 0xffffffffu;
  const unsigned ml = __reduce_min_sync(full, lo);
  return __hiloint2double((int)mh, (int)ml);
}
__device__ __forceinline__ void block_argmin_lazy(double& key, int& idx, int& exact, double (*red_val)[32],
                                                  int (*red_idx)[32], int& buf) {
  const unsigned full = 0xffffffffu;
  const unsigned tcode = ((unsigned)exact << 31) | (unsigned)idx; // equal keys: bounds first, then the index
  const unsigned hi = (unsigned)__double2hiint(key);
  const unsigned mh = __reduce_min_sync(full, hi);
  const unsigned lo = hi == mh ? (unsigned)__double2loint(key) : 0xffffffffu;
  const unsigned ml = __reduce_min_sync(full, lo);
  const unsigned mc = __reduce_min_sync(full, (hi == mh && lo == ml) ? tcode : 0xffffffffu);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) { red_val[buf][warp] = __hiloint2double((int)mh, (int)ml); red_idx[buf][warp] = (int)mc; }
  __syncthreads();
  double bk = red_val[buf][0];
  unsigned bc = (unsigned)red_idx[buf][0];
  for (int w = 1; w < nw; ++w) {
    const double ok = red_val[buf][w];
    const unsigned oc = (unsigned)red_idx[buf][w];
    if (ok < bk || (ok == bk && oc < bc)) { bk = ok; bc = oc; }
  }
  key = bk; idx = (int)(bc & 0x7fffffffu); exact = (int)(bc >> 31);
  buf ^= 1;
}
// smallest value of `v` (>= 0, +inf allowed) over the block
__device__ __forceinline__ double block_min_nonneg(double v, double (*red_val)[32], int& buf) {
  v = warp_min_nonneg(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) red_val[buf][warp] = v;
  __syncthreads();
  double bv = red_val[buf][0];
  for (int w = 1; w < nw; ++w) bv = fmin(bv, red_val[buf][w]);
  buf ^= 1;
  return bv;
}

// Lower bound of the pass-metric distance from p to a box, from the per-axis gaps d_k (0 inside the slab):
//   z^T M z >= z_k^2 / (M^-1)_kk >= d_k^2 / (M^-1)_kk   and   z^T M z >= lambda_min(M) |d|^2.
#ifndef BP_LAZY_GROW
#define BP_LAZY_GROW 3.0
#endif
struct PassBound {
  double c[3];      // (1 - eta) / (M^-1)_kk
  double lmin;      // (1 - eta) lambda_min(M)
};
__device__ __forceinline__ void pass_bound_init(const PassMetric& pm, PassBound* pb) {
  double M[9], Mi[9];
  bp_mat3_ata(pm.Q, M);
  const double det = bp_inv3(M, Mi);
  // lambda_min(M) = 1 / lambda_max(M^-1) >= 1 / ||M^-1||_F: a valid (at most sqrt(3) times weaker) bound without the
  // trigonometric eigenvalue solve, which cost every thread ~2.5 k cycles per pass
  double fro = 0.0;
#pragma unroll
  for (int k = 0; k < 9; ++k) fro += Mi[k] * Mi[k];
  const double lm = det > 0.0 ? 1.0 / sqrt(fro) : 0.0;
  // eta = 1e-3 covers the rounding of the inverse / eigenvalue up to cond(M) ~ 1e12; the bound only decides
  // WHICH closest-point QPs are solved, never a result
  const double keep = 1.0 - 1e-3;
  const bool ok = det > 0.0 && Mi[0] > 0.0 && Mi[4] > 0.0 && Mi[8] > 0.0;
  pb->c[0] = ok ? keep / Mi[0] : 0.0;
  pb->c[1] = ok ? keep / Mi[4] : 0.0;
  pb->c[2] = ok ? keep / Mi[8] : 0.0;
  pb->lmin = (lm > 0.0 && lm < BP_INF) ? keep * lm : 0.0;
}
__device__ __forceinline__ double box_dist_bound(const PassBound& pb, const double* p, const double* lb,
                                                 const double* ub) {
  const double d0 = fmax(fmax(lb[0] - p[0], p[0] - ub[0]), 0.0);
  const double d1 = fmax(fmax(lb[1] - p[1], p[1] - ub[1]), 0.0);
  const double d2 = fmax(fmax(lb[2] - p[2], p[2] - ub[2]), 0.0);
  const double q0 = d0 * d0, q1 = d1 * d1, q2 = d2 * d2;
  const double b2 = fmax(fmax(pb.c[0] * q0, pb.c[1] * q1), fmax(pb.c[2] * q2, pb.lmin * ((q0 + q1) + q2)));
  return sqrt(b2);
}

// ---------------------------------------------------------------------------
// General polytope obstacles (SURVEY 8f row 4): one WARP solves the closest-point QP of one polytope -- the
// candidates of bp_polytope_candidate (<= 1 + 15 + 105 + 455) are dealt to the lanes, the feasible candidate of
// least objective wins (first candidate number on ties, like the serial walk).  rows4: the polytope's rows
// staged in shared memory.  Every lane returns the same y; false: no feasible candidate (empty polytope).
// ---------------------------------------------------------------------------
struct SmemRows4 {
  const double* r;
  __device__ __forceinline__ double a(int i, int k) const { return r[4 * i + k]; }
  __device__ __forceinline__ double b(int i) const { return r[4 * i + 3]; }
};

__device__ __forceinline__ bool polytope_qp_warp(const BpPolyMetric& pmq, const double* rows4, int R, const double* p,
                                                 double* y) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  SmemRows4 rows{rows4};
  double best = BP_INF, yb[3] = {0.0, 0.0, 0.0}, yc[3], oc;
  int bidx = 0x7fffffff, cnt = 0;
#define BP_POLY_TRY(I, J, K)                                                                            \
  {                                                                                                     \
    if ((cnt & 31) == lane && bp_polytope_candidate(pmq, rows, R, p, (I), (J), (K), yc, &oc) && oc < best) { \
      best = oc; bidx = cnt; yb[0] = yc[0]; yb[1] = yc[1]; yb[2] = yc[2];                               \
    }                                                                                                   \
    ++cnt;                                                                                              \
  }
  BP_POLY_TRY(-1, -1, -1)
  for (int i = 0; i < R; ++i) BP_POLY_TRY(i, -1, -1)
  for (int i = 0; i < R; ++i)
    for (int j = i + 1; j < R; ++j) BP_POLY_TRY(i, j, -1)
  for (int i = 0; i < R; ++i)
    for (int j = i + 1; j < R; ++j)
      for (int k = j + 1; k < R; ++k) BP_POLY_TRY(i, j, k)
#undef BP_POLY_TRY
  const double bmin = warp_min_nonneg(best < 0.0 ? 0.0 : best);
  if (!(bmin < BP_INF)) return false;
  const unsigned cand = (best <= bmin) ? (unsigned)bidx : 0xffffffffu;    // (objectives are >= 0 up to rounding)
  const unsigned widx = __reduce_min_sync(full, cand);
  const int src = __ffs(__ballot_sync(full, cand == widx)) - 1;
  y[0] = __shfl_sync(full, yb[0], src);
  y[1] = __shfl_sync(full, yb[1], src);
  y[2] = __shfl_sync(full, yb[2], src);
  return true;
}

// min over the obstacle's vertices of a.v - b (vertex test of ConvexSetFinder.py:449-451 for a polytope)
__device__ __forceinline__ double poly_min_halfspace(const SceneView& sc, int j, const double* a, double bh) {
  const double* v = sc.verts + (size_t)j * sc.vmax * 3;
  const int nv = sc.nverts[j];
  double mn = BP_INF;
  for (int t = 0; t < nv; ++t) mn = fmin(mn, (a[0] * __ldg(v + 3 * t) + a[1] * __ldg(v + 3 * t + 1)) + a[2] * __ldg(v + 3 * t + 2) - bh);
  return mn;
}

#define BP_POLY_LIST 128

// One compute_polyhedron pass for the seed of this CTA (all threads call it): rows 6.. are written
// to Arow/brow (global or shared memory), *m_out = 6 + picks, *status_out = BP_OK / BP_ELLIPSE_VIOLATION.
//
// LAZY closest points: the greedy loop only ever needs the exact distance of the obstacle that is currently
// nearest; everything a picked halfspace cuts off dies by the vertex test, which needs no distance.  The table
// s_dist[j] therefore starts as a cheap LOWER BOUND of every distance (stored negated), and a box QP is solved
// only for entries whose bound does not exceed the best exact distance known.  The pick is the argmin over exact
// values once no bound is smaller or equal -- the same obstacle, the same bits as solving all N QPs (the QP of
// an entry is the same code on the same inputs whenever it runs).
// POLY: the obstacles are general polytopes (sc.rows != NULL): the bounds come from their bounding boxes, the exact
// closest points from warp-cooperative QPs over a shared work list, the vertex test walks their vertex lists.
template <bool POLY, int AW = 1>
__device__ __forceinline__ void poly_pass_point(const SceneView& sc, const PassMetric& pm, const double* p,
                                                double* s_dist, int cache_y, double (*red_val)[32],
                                                int (*red_idx)[32], double* Arow,
                                                double* brow, int m_max, int* m_out, int* status_out) {
  const int tid = threadIdx.x, T = blockDim.x;
  double* s_y = s_dist + sc.n;               // [3][N] when cache_y
  __shared__ int s_list[POLY ? BP_POLY_LIST : 1];
  __shared__ int s_nlist;
  __shared__ double s_prow[POLY ? 16 : 1][POLY ? BP_OBS_ROWS * 4 : 1];
  BpPolyMetric pmq;
  if (POLY) {
    double M9[9];
    bp_mat3_ata(pm.Q, M9);
    bp_poly_metric_init(M9, &pmq);
    if (tid == 0) s_nlist = 0;
  }
  BP_PPROF_MARK();
  PassBound pb;
  pass_bound_init(pm, &pb);
  // Entry k of this thread is obstacle j = tid + k T (k < 64 AW: N <= 64 AW T); `alive` has a bit per entry that
  // no picked halfspace has cut off yet, so the scans below touch live entries only.
  unsigned long long alive[AW];
#pragma unroll
  for (int w = 0; w < AW; ++w) alive[w] = 0ull;
  // phase 1: lower bounds (stored negated); a zero bound (p inside the box's slabs) is refined on the spot
  double lkey = BP_INF;
  int lidx = 0x3fffffff, lexact = 0;
  {
    int k = 0;
    for (int j = tid; j < sc.n; j += T, ++k) {
      double lb[3], ub[3];
      load_box(sc, j, lb, ub);
      double bd = box_dist_bound(pb, p, lb, ub);
      int ex = 0;
      if (POLY && !(bd > 0.0)) bd = DBL_MIN;        // inside the bounding box: a (useless) bound, refined on demand
      if (!(bd > 0.0)) {
        double y[3];
        bd = closest_on_box(pm, p, lb, ub, y);
        if (cache_y) { s_y[j] = y[0]; s_y[sc.n + j] = y[1]; s_y[2 * sc.n + j] = y[2]; }
        s_dist[j] = bd;
        ex = 1;
      } else {
        s_dist[j] = -bd;
      }
      alive[k >> 6] |= 1ull << (k & 63);
      if (bd < lkey || (bd == lkey && ex < lexact)) { lkey = bd; lidx = j; lexact = ex; }
    }
  }
  // (the barrier inside block_argmin_lazy orders these writes before the winner's point is read)

  // phase 2: greedy halfspaces
  int m_cur = 6;
  int status = BP_OK;
  int buf = 0;
  while (true) {
    double val = lkey;
    int idx = lidx, exact = lexact;
    if (buf == 0 && m_cur == 6) { BP_PPROF_LAP(0); } else { BP_PPROF_LAP(4); }
    block_argmin_lazy(val, idx, exact, red_val, red_idx, buf);
    BP_PPROF_LAP(1);
    if (!(val < BP_INF)) break;                      // no obstacle left
    if (!exact) {
      BP_PPROF_COUNT(6);
      // refine: every bound that could still beat (or tie with) the best exact distance -- and, to keep the
      // number of refinement rounds (one QP latency + one barrier each) small, everything within
      // BP_LAZY_GROW x the smallest bound: the next picks come from that shell
      double lex = BP_INF;
#pragma unroll
      for (int w = 0; w < AW; ++w)
        for (unsigned long long mk = alive[w]; mk; mk &= mk - 1) {
          const double d = s_dist[tid + (__ffsll((long long)mk) - 1 + 64 * w) * T];
          if (d >= 0.0) lex = fmin(lex, d);
        }
      const double ex = block_min_nonneg(lex, red_val, buf);
      const double thr = fmax(ex < BP_INF ? ex : 0.0, BP_LAZY_GROW * val);
      if (POLY) {
        // work list of the obstacles to refine (what does not fit waits for the next round)
#pragma unroll
        for (int w = 0; w < AW; ++w)
        for (unsigned long long mk = alive[w]; mk; mk &= mk - 1) {
          const int j = tid + (__ffsll((long long)mk) - 1 + 64 * w) * T;
          const double d = s_dist[j];
          if (d < 0.0 && -d <= thr) {
            const int slot = atomicAdd(&s_nlist, 1);
            if (slot < BP_POLY_LIST) s_list[slot] = j;
          }
        }
        __syncthreads();
        const int nl = s_nlist < BP_POLY_LIST ? s_nlist : BP_POLY_LIST;
        const int warp = tid >> 5, lane = tid & 31, nw = T >> 5;
        for (int q = warp; q < nl; q += nw) {
          const int j = s_list[q];
          const int R = sc.nrows[j];
          for (int e = lane; e < R * 4; e += 32) s_prow[warp][e] = __ldg(sc.rows + (size_t)j * BP_OBS_ROWS * 4 + e);
          __syncwarp();
          double y[3];
          const bool okq = polytope_qp_warp(pmq, s_prow[warp], R, p, y);
          if (lane == 0) {
            double d = BP_INF;                          // an empty polytope never constrains the set
            if (okq) {
              const double zz[3] = {y[0] - p[0], y[1] - p[1], y[2] - p[2]};
              double w[3];
              bp_mat3_vec(pm.Q, zz, w);
              d = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
            }
            s_dist[j] = d;
            if (cache_y) { s_y[j] = y[0]; s_y[sc.n + j] = y[1]; s_y[2 * sc.n + j] = y[2]; }
          }
          __syncwarp();
        }
        __syncthreads();
        if (tid == 0) s_nlist = 0;
      }
      lkey = BP_INF; lidx = 0x3fffffff; lexact = 0;
#pragma unroll
      for (int w = 0; w < AW; ++w)
      for (unsigned long long mk = alive[w]; mk; mk &= mk - 1) {
        const int j = tid + (__ffsll((long long)mk) - 1 + 64 * w) * T;
        double d = s_dist[j];
        int e = 1;
        if (d < 0.0) {
          if (!POLY && -d <= thr) {
            double lb[3], ub[3], y[3];
            load_box(sc, j, lb, ub);
            d = closest_on_box(pm, p, lb, ub, y);
            if (cache_y) { s_y[j] = y[0]; s_y[sc.n + j] = y[1]; s_y[2 * sc.n + j] = y[2]; }
            s_dist[j] = d;
          } else {
            d = -d;
            e = 0;
          }
        }
        if (!(d < BP_INF)) { alive[w] &= ~(1ull << (__ffsll((long long)mk) - 1)); continue; }   // empty polytope
        if (d < lkey || (d == lkey && e < lexact)) { lkey = d; lidx = j; lexact = e; }
      }
      BP_PPROF_LAP(2);
      continue;
    }
    BP_PPROF_COUNT(5);
    if (val < 0.99) { status = BP_ELLIPSE_VIOLATION; break; }   // :433-438
    double y[3];
    if (cache_y) {
      y[0] = s_y[idx]; y[1] = s_y[sc.n + idx]; y[2] = s_y[2 * sc.n + idx];
    } else if (POLY) {                         // large polytope scenes: warp 0 re-solves the winner's QP (same
      __shared__ double s_ywin[3];             // inputs, same candidate order, same bits) and hands it round
      if (tid < 32) {
        const int R = sc.nrows[idx];
        for (int e = tid; e < R * 4; e += 32) s_prow[0][e] = __ldg(sc.rows + (size_t)idx * BP_OBS_ROWS * 4 + e);
        __syncwarp();
        double yw[3] = {0.0, 0.0, 0.0};
        polytope_qp_warp(pmq, s_prow[0], R, p, yw);
        if (tid == 0) { s_ywin[0] = yw[0]; s_ywin[1] = yw[1]; s_ywin[2] = yw[2]; }
      }
      __syncthreads();
      y[0] = s_ywin[0]; y[1] = s_ywin[1]; y[2] = s_ywin[2];
      __syncthreads();                         // (s_prow[0] / s_ywin are reused by the next refinement round / pick)
    } else {                                   // large scenes: re-solve the winner's QP (same inputs, same bits)
      double lb[3], ub[3];
      load_box(sc, idx, lb, ub);
      closest_on_box(pm, p, lb, ub, y);
    }
    double zz[3] = {y[0] - p[0], y[1] - p[1], y[2] - p[2]};
    double a[3];
    bp_mat3_vec(pm.G, zz, a);
    a[0] *= 2.0; a[1] *= 2.0; a[2] *= 2.0;           // 2 (Q Q^T)(cp - p)   (:440)
    double bh = a[0] * y[0] + a[1] * y[1] + a[2] * y[2];
    double nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    a[0] /= nrm; a[1] /= nrm; a[2] /= nrm; bh /= nrm;
    if (tid == 0 && m_cur < m_max) {
      Arow[3 * m_cur + 0] = a[0]; Arow[3 * m_cur + 1] = a[1]; Arow[3 * m_cur + 2] = a[2];
      brow[m_cur] = bh;
    }
    ++m_cur;
    BP_PPROF_LAP(3);
    // delete the winner and every obstacle whose 8 vertices satisfy a.v - b >= -1e-4  (:447-458); live entries
    // are taken two at a time so that their box loads are in flight together
    lkey = BP_INF; lidx = 0x3fffffff; lexact = 0;
#pragma unroll
    for (int w = 0; w < AW; ++w)
    for (unsigned long long mk = alive[w]; mk;) {
      const int k0 = __ffsll((long long)mk) - 1;
      mk &= mk - 1;
      const int k1 = mk ? __ffsll((long long)mk) - 1 : k0;
      mk &= mk - 1;                               // (0 & anything stays 0)
      const int j0 = tid + (k0 + 64 * w) * T, j1 = tid + (k1 + 64 * w) * T;
      double l0[3], u0[3], l1[3], u1[3];
      load_box(sc, j0, l0, u0);
      load_box(sc, j1, l1, u1);
      const double d0 = s_dist[j0], d1 = s_dist[j1];
      const bool dead0 = j0 == idx || (POLY ? poly_min_halfspace(sc, j0, a, bh) : bp_box_min_halfspace(a, bh, l0, u0)) >= -1e-4;
      const bool dead1 = j1 == idx || (POLY ? poly_min_halfspace(sc, j1, a, bh) : bp_box_min_halfspace(a, bh, l1, u1)) >= -1e-4;
      if (dead0) alive[w] &= ~(1ull << k0);
      else {
        const int e = d0 >= 0.0;
        const double d = fabs(d0);
        if (d < lkey || (d == lkey && e < lexact)) { lkey = d; lidx = j0; lexact = e; }
      }
      if (k1 != k0) {
        if (dead1) alive[w] &= ~(1ull << k1);
        else {
          const int e = d1 >= 0.0;
          const double d = fabs(d1);
          if (d < lkey || (d == lkey && e < lexact)) { lkey = d; lidx = j1; lexact = e; }
        }
      }
    }
  }
  BP_PPROF_FLUSH();
  *m_out = m_cur;
  *status_out = status;
}

// ---------------------------------------------------------------------------
// compute_polyhedron pass for BOX scenes, "shell" form (same picks, same rows as poly_pass_point<false>):
//   A  every thread writes a cheap lower bound (squared, pass metric) of its obstacles' distances: key2[j];
//   B  the obstacles whose bound does not exceed thr = max(smallest exact distance known, GROW x smallest bound)
//      move into the SHELL (<= BP_SHELL slots in shared memory) and get their exact closest-point QP, one per
//      thread in parallel;
//   C  warp 0 alone runs the reference's greedy loop (ConvexSetFinder.py:431-458) over the shell while its
//      nearest entry is within thr -- every obstacle outside the shell is farther than thr, so the pick is the
//      global argmin (ties -> lowest obstacle index, quirk Q11): warp argmin by redux.sync, halfspace, vertex
//      test of the shell entries (boxes kept in the shell) -- no block barrier per pick;
//   D  all threads apply the new halfspaces to the obstacles outside the shell (vertex test, :447-458) and
//      recompute the smallest remaining bound; back to B until nothing is left.
// A pass costs 2-3 rounds of four barriers instead of two barriers per pick and per refinement round.
// Shell overflow (more than BP_SHELL obstacles within thr, e.g. a degenerate metric) -> *fallback = 1 and the
// caller reruns the pass with poly_pass_point.
// ---------------------------------------------------------------------------
// squared lower bound of the pass-metric distance from p to a box (see box_dist_bound)
__device__ __forceinline__ double box_bound2(const PassBound& pb, const double* p, const double* lb, const double* ub) {
  const double d0 = fmax(fmax(lb[0] - p[0], p[0] - ub[0]), 0.0);
  const double d1 = fmax(fmax(lb[1] - p[1], p[1] - ub[1]), 0.0);
  const double d2 = fmax(fmax(lb[2] - p[2], p[2] - ub[2]), 0.0);
  const double q0 = d0 * d0, q1 = d1 * d1, q2 = d2 * d2;
  return fmax(fmax(pb.c[0] * q0, pb.c[1] * q1), fmax(pb.c[2] * q2, pb.lmin * ((q0 + q1) + q2)));
}
// smallest value (>= 0, +inf allowed) and the sum of an int over the block
__device__ __forceinline__ double block_min_count(double v, int& cnt, double (*red_val)[32], int (*red_cnt)[32],
                                                  int& buf) {
  v = warp_min_nonneg(v);
  const int c = __reduce_add_sync(0xffffffffu, cnt);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) { red_val[buf][warp] = v; red_cnt[buf][warp] = c; }
  __syncthreads();
  double bv = red_val[buf][0];
  int bc = red_cnt[buf][0];
  for (int w = 1; w < nw; ++w) { bv = fmin(bv, red_val[buf][w]); bc += red_cnt[buf][w]; }
  buf ^= 1;
  cnt = bc;
  return bv;
}

#define BP_SHELL 128
struct ShellMem {
  double dist[BP_SHELL];               // exact distance (:429); +inf = free slot
  double y[3][BP_SHELL];               // closest point on the obstacle
  double lb[3][BP_SHELL], ub[3][BP_SHELL];
  double pick[BP_MAX_ROWS][4];         // halfspaces picked since the last sweep over the obstacles outside the shell
  double exmin;                        // smallest exact distance left in the shell
  int idx[BP_SHELL];                   // obstacle index of a slot
  int free_list[BP_SHELL];             // free slots
  int new_list[BP_SHELL];              // slots filled in this round (exact QP pending)
  int n_free, cnt, n_pick, m_cur, status, pad_;
  int hist[8][16];                     // per-warp counts of the obstacles within the candidate thresholds
};

template <int AW>
__device__ __forceinline__ void poly_pass_shell(const SceneView& sc, const PassMetric& pm, const double* p,
                                                double* s_key, ShellMem* sh, double (*red_val)[32],
                                                int (*red_idx)[32], double* Arow, double* brow, int m_max, int* m_out,
                                                int* status_out, int* fallback) {
  const unsigned full = 0xffffffffu;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  BP_PPROF_MARK();
  PassBound pb;
  pass_bound_init(pm, &pb);
  unsigned long long alive[AW];
#pragma unroll
  for (int w = 0; w < AW; ++w) alive[w] = 0ull;
  // ---- A: squared lower bounds of every obstacle (entry k of this thread is obstacle tid + k T)
  double lmin2 = BP_INF;
  int n_alive = 0;
  {
    // two obstacles per trip: their loads and the two short dependency chains overlap
    int k = 0;
    for (int j = tid; j < sc.n; j += 2 * T, k += 2) {
      const int j1 = j + T;
      const bool two = j1 < sc.n;
      double la[3], ua[3], lc[3], uc[3];
      load_box(sc, j, la, ua);
      load_box(sc, two ? j1 : j, lc, uc);
      const double ba = box_bound2(pb, p, la, ua), bc = box_bound2(pb, p, lc, uc);
      s_key[j] = ba;
      alive[k >> 6] |= 1ull << (k & 63);
      lmin2 = fmin(lmin2, ba);
      ++n_alive;
      if (two) {
        s_key[j1] = bc;
        alive[(k + 1) >> 6] |= 1ull << ((k + 1) & 63);
        lmin2 = fmin(lmin2, bc);
        ++n_alive;
      }
    }
  }
  for (int e = tid; e < BP_SHELL; e += T) { sh->dist[e] = BP_INF; sh->free_list[e] = e; }
  if (tid == 0) { sh->n_free = BP_SHELL; sh->cnt = 0; sh->n_pick = 0; sh->m_cur = 6; sh->status = BP_OK; sh->exmin = BP_INF; }
  int buf = 0;
  int m_cur = 6, status = BP_OK;
  BP_PPROF_LAP(0);
  while (true) {
    // smallest bound outside the shell (the barrier inside also publishes the shell state written by warp 0)
    int n_out = n_alive;
    const double bmin2 = block_min_count(lmin2, n_out, red_val, red_idx, buf);
    const double exmin = sh->exmin;
    if (!(bmin2 < BP_INF) && !(exmin < BP_INF)) break;                 // no obstacle left
    BP_PPROF_COUNT(6);
    // ---- B: move the obstacles within thr into the shell; once everything left outside fits, take it all
    // (one more round ends the pass)
    const int n_free = sh->n_free;
    double thr = BP_INF, thr2 = BP_INF;
    if (bmin2 < BP_INF && n_out > n_free) {
      // Every round costs one closest-point QP latency however few QPs it solves, so the shell is filled as far
      // as it goes: the widest of the thresholds GROW x {1, 2, 4, 8} x (smallest bound) that still fits.
      // (a dense neighbourhood where not even GROW x fits gets a second, finer ladder below GROW x)
      const double bmin = sqrt(bmin2), floor_ = exmin < BP_INF ? exmin : 0.0;
      for (int level = 0; level < 2; ++level) {
        // level 0: GROW x 1.4^g (the count grows about cubically with the radius: a ladder this fine fills the
        // shell to more than a third); level 1: eight steps between 1 x and GROW x
        double cand[8], cand2[8];
        int c8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        double f = level == 0 ? BP_LAZY_GROW : 1.0 + (BP_LAZY_GROW - 1.0) * 0.06;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          cand[g] = fmax(floor_, f * bmin);
          cand2[g] = cand[g] * cand[g];
          f = level == 0 ? f * 1.4 : f + (BP_LAZY_GROW - 1.0) * 0.12;
        }
#pragma unroll
        for (int w = 0; w < AW; ++w)
          for (unsigned long long mk = alive[w]; mk; mk &= mk - 1) {
            const double key = s_key[tid + (__ffsll((long long)mk) - 1 + 64 * w) * T];
#pragma unroll
            for (int g = 0; g < 8; ++g) c8[g] += key <= cand2[g];
          }
        if (level == 1) __syncthreads();                 // the level-0 counts have been read by everybody
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const int c = __reduce_add_sync(full, c8[g]);
          if (lane == 0) sh->hist[g][warp] = c;
        }
        __syncthreads();
        int pick_g = -1;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          int tot = 0;
          for (int w = 0; w < (T >> 5); ++w) tot += sh->hist[g][w];
          if (tot <= n_free) pick_g = g;
        }
        thr = cand[pick_g < 0 ? 0 : pick_g];
        thr2 = cand2[pick_g < 0 ? 0 : pick_g];
        if (pick_g >= 0) break;                          // (else: the finer ladder; after it the retry below)
      }
    }
    unsigned long long taken[AW];
#pragma unroll
    for (int w = 0; w < AW; ++w) taken[w] = 0ull;
    bool over = false;
    for (int attempt = 0; attempt < 2; ++attempt) {
      if (bmin2 < BP_INF) {
#pragma unroll
        for (int w = 0; w < AW; ++w) {
          taken[w] = 0ull;
          for (unsigned long long mk = alive[w]; mk; mk &= mk - 1) {
            const int k = __ffsll((long long)mk) - 1;
            const int j = tid + (k + 64 * w) * T;
            if (s_key[j] <= thr2) {
              const int slot = atomicAdd(&sh->cnt, 1);
              if (slot < n_free) { const int ph = sh->free_list[slot]; sh->idx[ph] = j; sh->new_list[slot] = ph; }
              taken[w] |= 1ull << k;
            }
          }
        }
      }
      __syncthreads();
      over = sh->cnt > n_free;
      if (!over) break;
      __syncthreads();                                   // everybody has read cnt
      if (tid == 0) sh->cnt = 0;
      // too many obstacles within GROW x the smallest bound: take only what the next pick needs
      thr = fmax(exmin < BP_INF ? exmin : 0.0, sqrt(bmin2));
      thr2 = fmax(thr * thr, bmin2);
      __syncthreads();
    }
    if (over) { BP_PPROF_FLUSH(); *fallback = 1; return; }
    const int n_new = sh->cnt;
    BP_PPROF_ADDN(7, n_new);
#pragma unroll
    for (int w = 0; w < AW; ++w) alive[w] &= ~taken[w];
    // exact closest points of the new shell entries
    for (int e = tid; e < n_new; e += T) {
      const int ph = sh->new_list[e];
      const int j = sh->idx[ph];
      double lb[3], ub[3], y[3];
      load_box(sc, j, lb, ub);
      const double d = closest_on_box(pm, p, lb, ub, y);
      sh->dist[ph] = d;
#pragma unroll
      for (int c = 0; c < 3; ++c) { sh->y[c][ph] = y[c]; sh->lb[c][ph] = lb[c]; sh->ub[c][ph] = ub[c]; }
    }
    __syncthreads();
    BP_PPROF_LAP(2);
    // ---- C: greedy picks over the shell, warp 0
    if (warp == 0) {
      double d[BP_SHELL / 32];
      int id[BP_SHELL / 32];
#pragma unroll
      for (int q = 0; q < BP_SHELL / 32; ++q) { d[q] = sh->dist[lane + 32 * q]; id[q] = sh->idx[lane + 32 * q]; }
      int m = m_cur, npick = 0, st = BP_OK;
      while (npick < BP_MAX_ROWS) {
        double lv = d[0];
        int li = id[0], lq = 0;
#pragma unroll
        for (int q = 1; q < BP_SHELL / 32; ++q)
          if (d[q] < lv || (d[q] == lv && id[q] < li)) { lv = d[q]; li = id[q]; lq = q; }
        // warp argmin of non-negative doubles: order of the bit patterns, then the obstacle index
        const unsigned hi = (unsigned)__double2hiint(lv);
        const unsigned mh = __reduce_min_sync(full, hi);
        const unsigned lo = hi == mh ? (unsigned)__double2loint(lv) : 0xffffffffu;
        const unsigned ml = __reduce_min_sync(full, lo);
        const bool cand = hi == mh && lo == ml && lv < BP_INF;
        const unsigned mc = __reduce_min_sync(full, cand ? (unsigned)li : 0xffffffffu);
        const double val = __hiloint2double((int)mh, (int)ml);
        if (!(val < BP_INF) || !(val <= thr)) break;            // shell exhausted / the rest needs a wider shell
        BP_PPROF_COUNT(5);
        if (val < 0.99) { st = BP_ELLIPSE_VIOLATION; break; }   // :433-438
        const int src = __ffs(__ballot_sync(full, cand && (unsigned)li == mc)) - 1;
        const int e = __shfl_sync(full, lane + 32 * lq, src);
        const double y[3] = {sh->y[0][e], sh->y[1][e], sh->y[2][e]};
        double zz[3] = {y[0] - p[0], y[1] - p[1], y[2] - p[2]};
        double a[3];
        bp_mat3_vec(pm.G, zz, a);
        a[0] *= 2.0; a[1] *= 2.0; a[2] *= 2.0;           // 2 (Q Q^T)(cp - p)   (:440)
        double bh = a[0] * y[0] + a[1] * y[1] + a[2] * y[2];
        const double inrm = rsqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);   // a / ||a||, b / ||a||  (:441-444)
        a[0] *= inrm; a[1] *= inrm; a[2] *= inrm; bh *= inrm;
        if (lane == 0) {
          if (m < m_max) { Arow[3 * m + 0] = a[0]; Arow[3 * m + 1] = a[1]; Arow[3 * m + 2] = a[2]; brow[m] = bh; }
          sh->pick[npick][0] = a[0]; sh->pick[npick][1] = a[1]; sh->pick[npick][2] = a[2]; sh->pick[npick][3] = bh;
        }
        ++m; ++npick;
        // delete the winner and every shell obstacle whose 8 vertices satisfy a.v - b >= -1e-4  (:447-458)
#pragma unroll
        for (int q = 0; q < BP_SHELL / 32; ++q) {
          if (d[q] < BP_INF) {
            const int s = lane + 32 * q;
            const double l3[3] = {sh->lb[0][s], sh->lb[1][s], sh->lb[2][s]};
            const double u3[3] = {sh->ub[0][s], sh->ub[1][s], sh->ub[2][s]};
            if ((unsigned)id[q] == mc || bp_box_min_halfspace(a, bh, l3, u3) >= -1e-4) d[q] = BP_INF;
          }
        }
      }
      // shell bookkeeping for the next round: free slots, smallest exact distance left
      int nf = 0;
      double ex = BP_INF;
#pragma unroll
      for (int q = 0; q < BP_SHELL / 32; ++q) {
        const bool fr = !(d[q] < BP_INF);
        const unsigned bal = __ballot_sync(full, fr);
        if (fr) { sh->free_list[nf + __popc(bal & ((1u << lane) - 1u))] = lane + 32 * q; sh->dist[lane + 32 * q] = BP_INF; }
        else ex = fmin(ex, d[q]);
        nf += __popc(bal);
      }
      ex = warp_min_nonneg(ex);
      if (lane == 0) { sh->n_free = nf; sh->cnt = 0; sh->n_pick = npick; sh->m_cur = m; sh->status = st; sh->exmin = ex; }
    }
    __syncthreads();
    BP_PPROF_LAP(3);
    m_cur = sh->m_cur;
    status = sh->status;
    if (status != BP_OK) break;
    // ---- D: the new halfspaces against the obstacles outside the shell
    const int npk = sh->n_pick;
    lmin2 = BP_INF;
    n_alive = 0;
#pragma unroll
    for (int w = 0; w < AW; ++w) {
      for (unsigned long long mk = alive[w]; mk; mk &= mk - 1) {
        const int k = __ffsll((long long)mk) - 1;
        const int j = tid + (k + 64 * w) * T;
        bool dead = false;
        if (npk > 0) {
          double lb[3], ub[3];
          load_box(sc, j, lb, ub);
          for (int t = 0; t < npk && !dead; ++t) {
            // min over the 8 vertices of a.v - b: by monotone rounding min(a lb, a ub) == a * (a >= 0 ? lb : ub),
            // the same bits as bp_box_min_halfspace with half the FP64 instructions
            const double a0 = sh->pick[t][0], a1 = sh->pick[t][1], a2 = sh->pick[t][2];
            const double t0 = a0 * (a0 >= 0.0 ? lb[0] : ub[0]);
            const double t1 = a1 * (a1 >= 0.0 ? lb[1] : ub[1]);
            const double t2 = a2 * (a2 >= 0.0 ? lb[2] : ub[2]);
            dead = (((t0 + t1) + t2) - sh->pick[t][3]) >= -1e-4;
          }
        }
        if (dead) alive[w] &= ~(1ull << k);
        else { lmin2 = fmin(lmin2, s_key[j]); ++n_alive; }
      }
    }
    BP_PPROF_LAP(4);
  }
  BP_PPROF_FLUSH();
  *m_out = m_cur;
  *status_out = status;
}

// (arguments by value: taking the address of the caller's metric / scene view would move them to local memory
// on the hot path as well)
struct PassResult { int m, status; };
__device__ unsigned long long g_shell_fallbacks;     // passes that overflowed the shell (bp_debug_counters)
template <int AW>
__device__ __noinline__ PassResult poly_pass_point_fallback(SceneView sc, PassMetric pm, Vec3 p, double* s_dist,
                                                            double (*red_val)[32], int (*red_idx)[32], double* Arow,
                                                            double* brow, int m_max) {
  PassResult r;
  if (threadIdx.x == 0) atomicAdd(&g_shell_fallbacks, 1ull);
  poly_pass_point<false, AW>(sc, pm, p.v, s_dist, 0, red_val, red_idx, Arow, brow, m_max, &r.m, &r.status);
  return r;
}

// one compute_polyhedron pass of this CTA's seed: box scenes take the shell form (AW words of alive bits per
// thread: N <= 64 AW blockDim.x), polytope scenes the lazy per-pick form
template <bool POLY, int AW>
__device__ __forceinline__ void poly_pass(const SceneView& sc, int n_max, const PassMetric& pm, const double* p,
                                          double* s_dist, int cache_y, double (*red_val)[32], int (*red_idx)[32],
                                          double* Arow, double* brow, int m_max, int* m_out, int* status_out) {
  if (POLY) {
    poly_pass_point<true>(sc, pm, p, s_dist, cache_y, red_val, red_idx, Arow, brow, m_max, m_out, status_out);
  } else {
    ShellMem* sh = (ShellMem*)(s_dist + ((n_max + 1) & ~1));
    int fb = 0;
    poly_pass_shell<AW>(sc, pm, p, s_dist, sh, red_val, red_idx, Arow, brow, m_max, m_out, status_out, &fb);
    if (fb) {                                  // (block-uniform) shell overflow: the per-pick form, from scratch
      __syncthreads();
      Vec3 pv;
      pv.v[0] = p[0]; pv.v[1] = p[1]; pv.v[2] = p[2];
      const PassResult r = poly_pass_point_fallback<AW>(sc, pm, pv, s_dist, red_val, red_idx, Arow, brow, m_max);
      *m_out = r.m;
      *status_out = r.status;
    }
  }
}

template <bool POLY>
__global__ void __launch_bounds__(512) k_poly_point(SceneView sc_all, PolyParams pr) {
  const SceneView sc = scene_of_item(sc_all, blockIdx.x);
  extern __shared__ double s_dist[];
  __shared__ double red_val[2][32];
  __shared__ int red_idx[2][32];
  const int s = blockIdx.x;
  const int tid = threadIdx.x, T = blockDim.x;
  double p[3];
  PassMetric pm;
  double* Arow = pr.A + (size_t)s * pr.m_max * 3;
  double* brow = pr.b + (size_t)s * pr.m_max;
  if (pr.mode == 1) {
    SeedState* st = pr.state + s;
    if (!st->active || st->status != BP_OK) return;
    // while |det - det_old| / det_old > 0.01: k += 1; if k > max_iter: break   (:203-207)
    double det = st->det, det_old = st->det_old;
    int k = st->k;
    bool go = fabs(det - det_old) / det_old > 0.01;
    if (go) go = (k + 1 <= pr.max_iter);
    __syncthreads();                       // everybody has read the state
    if (!go) {
      if (tid == 0) { st->active = 0; if (fabs(det - det_old) / det_old > 0.01) st->k = k + 1; }
      return;
    }
    if (tid == 0) st->k = k + 1;
#pragma unroll
    for (int q = 0; q < 3; ++q) p[q] = st->p[q];
    pass_metric_init(st->Q, &pm);
    if (tid < 6) {
      int ax = tid >> 1;
      double sgn = (tid & 1) ? -1.0 : 1.0;
      Arow[3 * tid + 0] = ax == 0 ? sgn : 0.0;
      Arow[3 * tid + 1] = ax == 1 ? sgn : 0.0;
      Arow[3 * tid + 2] = ax == 2 ? sgn : 0.0;
      brow[tid] = pr.ws_rows[tid];
    }
  } else {
#pragma unroll
    for (int q = 0; q < 3; ++q) p[q] = pr.seeds[(size_t)s * 3 + q];
    double Q[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) Q[q] = pr.q_ellipse[(size_t)s * 9 + q];
    pass_metric_init(Q, &pm);
    if (tid < 6) {
      const double* r = pr.init_rows + ((size_t)s * 6 + tid) * 4;
      Arow[3 * tid + 0] = r[0]; Arow[3 * tid + 1] = r[1]; Arow[3 * tid + 2] = r[2];
      brow[tid] = r[3];
    }
  }

  int m_cur, status;
  if (POLY || pr.shell)
    poly_pass<POLY, 1>(sc, sc_all.n, pm, p, s_dist, pr.cache_y, red_val, red_idx, Arow, brow, pr.m_max, &m_cur, &status);
  else     // the largest scenes: only the distance table fits in shared memory
    poly_pass_point<false, 1>(sc, pm, p, s_dist, 0, red_val, red_idx, Arow, brow, pr.m_max, &m_cur, &status);
  if (status == BP_OK && m_cur > pr.m_max) status = BP_ROW_OVERFLOW;
  // rows past the last one keep the padding of normalize_set_size (A = 0, b = 10): an earlier,
  // longer pass may have left its rows there
  for (int r = m_cur + tid; r < pr.m_max; r += T) {
    Arow[3 * r] = 0.0; Arow[3 * r + 1] = 0.0; Arow[3 * r + 2] = 0.0;
    brow[r] = 10.0;
  }
  if (tid == 0) {
    pr.m[s] = m_cur < pr.m_max ? m_cur : pr.m_max;
    if (pr.mode == 1) {
      if (status == BP_OK && pr.row_cap > 0 && m_cur > pr.row_cap) status = BP_ROW_CAP;
      if (status != BP_OK) { pr.state[s].status = status; pr.state[s].active = 0; }
      if (m_cur > pr.state[s].rows_peak) pr.state[s].rows_peak = m_cur;
    } else {
      pr.status[s] = status;
    }
  }
}

// ---------------------------------------------------------------------------
// K5 fused: the whole find_set_around_point loop (ConvexSetFinder.py:190-240) for one seed in one
// persistent CTA of 128 threads: polyhedron pass (all threads) -> MVIE (warp 0, rows in shared
// memory) -> loop tests, up to max_iter times, + the trailing free-centre MVIE.  Compared with the
// (k_poly_point, k_mvie) launch sequence every seed advances at its own pace: a pass no longer waits
// for the slowest MVIE of the whole batch, and the rows never leave shared memory between the phases.
// Used for scenes whose distance table leaves room for two CTAs per SM (N <= 4096).
// ---------------------------------------------------------------------------
// Exact axis-aligned bounding box of the polytope {A x <= b} (ms rows) by vertex enumeration over all row
// triples, by the 128 threads of a CTA; rows may live in global or shared memory.  out6 = lo[3] | hi[3]
// (-inf / +inf when the description is unbounded or has no vertex -- never reject on such a set).
// Used by k_set_aabb and by the epilogue of the fused set build (same code, same bits).
#define BP_AABB_EPS 1e-9
__device__ __forceinline__ void cta_set_aabb(const double* As, const double* bs, int ms, double (*red)[6],
                                             double* out6) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double lo[3] = {BP_INF, BP_INF, BP_INF}, hi[3] = {-BP_INF, -BP_INF, -BP_INF};
  // all row triples (i < j < k), flattened over the threads so that every thread walks the same number of
  // candidates (the nested-loop version ran at 8.7 active threads/warp)
  const int ntrip = ms * (ms - 1) * (ms - 2) / 6;
  for (int t = threadIdx.x; t < ntrip; t += 128) {
    int i = 0, rem = t;
    for (;;) { const int c = (ms - 1 - i) * (ms - 2 - i) / 2; if (rem < c) break; rem -= c; ++i; }
    int j = i + 1;
    for (;;) { const int c = ms - 1 - j; if (rem < c) break; rem -= c; ++j; }
    const int k = j + 1 + rem;
    const double a0 = As[3 * i], a1 = As[3 * i + 1], a2 = As[3 * i + 2], ab = bs[i];
    const double c0 = As[3 * j], c1 = As[3 * j + 1], c2 = As[3 * j + 2], cb = bs[j];
    const double d0 = As[3 * k], d1 = As[3 * k + 1], d2 = As[3 * k + 2], db = bs[k];
    const double n0 = a1 * c2 - a2 * c1, n1 = a2 * c0 - a0 * c2, n2 = a0 * c1 - a1 * c0;      // a x c
    const double det = n0 * d0 + n1 * d1 + n2 * d2;
    const double scale = (fabs(n0) + fabs(n1) + fabs(n2)) * (fabs(d0) + fabs(d1) + fabs(d2));
    if (!(fabs(det) > 1e-12 * scale)) continue;
    // v = (ab (c x d) + cb (d x a) + db (a x c)) / det
    const double e0 = c1 * d2 - c2 * d1, e1 = c2 * d0 - c0 * d2, e2 = c0 * d1 - c1 * d0;
    const double f0 = d1 * a2 - d2 * a1, f1 = d2 * a0 - d0 * a2, f2 = d0 * a1 - d1 * a0;
    const double id = 1.0 / det;
    const double v0 = (ab * e0 + cb * f0 + db * n0) * id;
    const double v1 = (ab * e1 + cb * f1 + db * n1) * id;
    const double v2 = (ab * e2 + cb * f2 + db * n2) * id;
    bool inside = true;
    for (int r = 0; r < ms; ++r) {
      const double q0 = As[3 * r], q1 = As[3 * r + 1], q2 = As[3 * r + 2];
      const double viol = q0 * v0 + q1 * v1 + q2 * v2 - bs[r];
      if (viol > BP_AABB_EPS * (1.0 + fabs(q0 * v0) + fabs(q1 * v1) + fabs(q2 * v2))) inside = false;
    }
    if (inside) {
      lo[0] = fmin(lo[0], v0); hi[0] = fmax(hi[0], v0);
      lo[1] = fmin(lo[1], v1); hi[1] = fmax(hi[1], v1);
      lo[2] = fmin(lo[2], v2); hi[2] = fmax(hi[2], v2);
    }
  }
  // A set with a vertex can still be unbounded (a cone, a prism closed at one end): the box of its vertices would
  // then be too small, and the pre-tests would reject pairs that meet the set away from them.  Such a set has a
  // recession direction d != 0 with A d <= 0; when the rows span R^3 (else there is no vertex) that cone is pointed
  // and has an extreme ray d = +-(a_i x a_j), so every row pair is tried.  The test is loose on purpose: a set that
  // is bounded only to within rounding loses its box, which costs the pre-tests and never a pair.
  bool ray = false;
  const int npair = ms * (ms - 1) / 2;
  for (int t = threadIdx.x; t < npair && !ray; t += 128) {
    int i = 0, rem = t;
    for (;;) { const int c = ms - 1 - i; if (rem < c) break; rem -= c; ++i; }
    const int j = i + 1 + rem;
    const double a0 = As[3 * i], a1 = As[3 * i + 1], a2 = As[3 * i + 2];
    const double c0 = As[3 * j], c1 = As[3 * j + 1], c2 = As[3 * j + 2];
    const double d0 = a1 * c2 - a2 * c1, d1 = a2 * c0 - a0 * c2, d2 = a0 * c1 - a1 * c0;
    const double dd = d0 * d0 + d1 * d1 + d2 * d2;
    if (!(dd > 1e-24 * (a0 * a0 + a1 * a1 + a2 * a2) * (c0 * c0 + c1 * c1 + c2 * c2))) continue;   // parallel rows
    bool pos = true, neg = true;                          // A d <= 0 / A (-d) <= 0, up to rounding
    for (int r = 0; r < ms && (pos || neg); ++r) {
      const double q0 = As[3 * r], q1 = As[3 * r + 1], q2 = As[3 * r + 2];
      const double q = q0 * d0 + q1 * d1 + q2 * d2;
      const double lim = BP_AABB_EPS * (fabs(q0 * d0) + fabs(q1 * d1) + fabs(q2 * d2));
      if (q > lim) pos = false;
      if (-q > lim) neg = false;
    }
    ray = pos || neg;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      lo[k] = fmin(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], off));
      hi[k] = fmax(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], off));
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { red[warp][k] = lo[k]; red[warp][3 + k] = hi[k]; }
  }
  const int unbounded = __syncthreads_or(ray);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 4; ++w) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { lo[k] = fmin(lo[k], red[w][k]); hi[k] = fmax(hi[k], red[w][3 + k]); }
    }
    const bool none = !(lo[0] <= hi[0]) || unbounded;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      out6[k] = none ? -BP_INF : lo[k];
      out6[3 + k] = none ? BP_INF : hi[k];
    }
  }
}

// where the owner of a set also delivers it (multi-GPU exchange by peer stores, SURVEY 8e)
struct PeerTables {
  const unsigned long long* base;   // device array [world]: base address of every rank's symmetric allocation
  int world, slot0;                 // this rank's sets go to rows slot0 .. slot0 + S - 1 of the global tables
  size_t off_A, off_b, off_m, off_aabb;
};

// Pair tests in the tail of the set build ("finished CTAs become pair workers", section 7 of DESIGN.md): a CTA whose
// set is finished publishes an arrival flag and then tests its set against every set that arrives AFTER it, so
// that when the last set of the whole job arrives only its own pairs are left -- one per waiting CTA.
struct TailParams {
  int S;                     // number of sets in the (global) tables; 0: no tail work
  int words;                 // adjacency words per row
  const double* A;           // LOCAL copies of the tables [S,m_max,3] | [S,m_max] | [S] | [S,6]
  const double* b;
  const int* m;
  const double* aabb;
  unsigned int* count;       // arrival counter of this rank's log (S per step, never reset)
  unsigned long long* log;   // [S] ring of (epoch << 32 | set id)
  unsigned int* bits;        // [2][S][words] adjacency, double-buffered by the parity of the epoch (multi-GPU)
  const int* epoch;          // device int, bumped by bp_step_begin
  size_t off_count, off_log, off_bits;   // byte offsets in every rank's symmetric allocation
  double tol;
};
#define BP_TAIL_WORK_DOUBLES (4 * (BP_LP_SCRATCH_DOUBLES + 2 * (BP_MAX_ROWS * 4 + 8)))
__device__ void fused_tail_pairs(TailParams tp, PeerTables peers, int g, int m_max, const double* my_box, double* work);

struct FusedParams {
  TailParams tail;
  double* aabb;              // [S,6] or NULL: exact bounding box of every finished set (what k_set_aabb computes)
  PeerTables peers;          // peers.world > 0: finished sets and boxes are also stored into every rank's tables
  const double* seeds;       // [S,3] seeds (MODE 0) / segment starts p0 (MODE 1)
  const double* dp1;         // [S,3] segment vectors (MODE 1)
  double ws_rows[6];
  double* A;
  double* b;
  int* m;
  double* q_ellipse;
  double* p_mid;
  int* status;
  int* iters;
  int* rows_peak;
  int m_max, max_iter, fixed_mid, optimize, row_cap, cache_y;
  int stage;                 // box scene: stage the scene columns in shared memory (TMA) after key table + shell
  int spec;                  // trailing free-centre solve speculatively next to EVERY pass's fixed-centre solve
};

struct GlobalRows {
  const double* A;
  const double* B;
  __device__ __forceinline__ double a(int i, int k) const { return __ldg(A + 3 * i + k); }
  __device__ __forceinline__ double b(int i) const { return __ldg(B + i); }
};


struct SharedRows {
  const double* A;
  const double* B;
  __device__ __forceinline__ double a(int i, int k) const { return A[3 * i + k]; }
  __device__ __forceinline__ double b(int i) const { return B[i]; }
};

// MODE 0: find_set_around_point (:190-240).  MODE 1: find_set_around_line (:242-307) -- the same loop around
// the midpoint of the segment p0 .. p0 + dp1 with the fixed-rotation MVIE (mvie_socp_fixed_r); no trailing MVIE,
// and with optimize == 0 one free-centre MVIE after the first pass (:278-282).
__device__ unsigned g_sm_slot[256];     // CTAs started per SM (only its parity is used, never reset)

// SPEC: the instantiation with the speculative trailing solve (and the second, abortable copy of the free-centre
// solver); the plain one is what every launch without waves over a large scene runs.
template <int MODE, bool POLY, int AW = 1, bool SPEC = false>
__global__ void __launch_bounds__(128) k_iris_fused(SceneView sc_all, FusedParams pr) {
  SceneView sc = scene_of_item(sc_all, blockIdx.x);
  extern __shared__ __align__(16) double s_dist[];
  __shared__ double red_val[2][32];
  __shared__ int red_idx[2][32];
  __shared__ double sA[BP_MAX_ROWS * 3], sb[BP_MAX_ROWS];
  __shared__ double scratch[BP_MVIE_SCRATCH_DOUBLES];
  __shared__ double scratch2[MODE == 0 ? BP_MVIE_SCRATCH_DOUBLES : 1];   // the concurrent trailing solve (below)
  __shared__ __align__(8) uint64_t stage_bar;
  if (!POLY && pr.stage && (((uintptr_t)sc.lb[0] | (uintptr_t)sc.lb[1]) & 15) == 0) {
    // (a segment of a scene batch that starts at an odd obstacle index is not 16-byte aligned: global loads then)
    double* s_scene = s_dist + ((sc_all.n + 1) & ~1) + 2 * ((sizeof(ShellMem) + 15) / 16);
    sc = stage_scene(sc, s_scene, &stage_bar);
  }
  __shared__ double c_Q[9], c_p[3], c_det;
  __shared__ double f_Q[9], f_p[3];
  __shared__ int c_status, c_small, f_status, c_mw, f_done;
  __shared__ volatile int c_abort;
  const int s = blockIdx.x, tid = threadIdx.x;
#ifdef BPGEO_PROFILE
  const long long prof_k0_ = clock64();
#endif
  // The MVIE is a one-warp solve.  Two CTAs share an SM, and a warp's scheduler (SM sub-partition) is its index
  // mod 4: the CTAs of an SM take their slot from a per-SM counter so that their solver warps -- primary 2 slot,
  // the concurrent trailing solve 2 slot + 1 -- sit on four different sub-partitions and never share an FP64 pipe.
  if (tid == 0) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    c_mw = (int)((atomicAdd(&g_sm_slot[smid & 255u], 1u) & 1u) << 1);
  }
  __syncthreads();
  const int warp_id = tid >> 5, mw = c_mw, mw2 = c_mw + 1;
  bool have_final = false;
  double Q[9] = {1e4, 0, 0, 0, 1e4, 0, 0, 0, 1e4};          // q_ellipse = diag(1/1e-4) (:192-194)
  double p[3] = {pr.seeds[3 * (size_t)s], pr.seeds[3 * (size_t)s + 1], pr.seeds[3 * (size_t)s + 2]};
  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  double a_lb = 0.0;
  if (MODE == 1) {                                            // :243-261
    const double dp1[3] = {pr.dp1[3 * (size_t)s], pr.dp1[3 * (size_t)s + 1], pr.dp1[3 * (size_t)s + 2]};
    const double p1[3] = {p[0] + dp1[0], p[1] + dp1[1], p[2] + dp1[2]};
    double l_seg;
    bp_line_frame(dp1, R, &l_seg);
#pragma unroll
    for (int q = 0; q < 3; ++q) p[q] = (p[q] + p1[q]) / 2;
    a_lb = l_seg * l_seg / 4;
    const double y0[3] = {a_lb, 1e-4, 1e-4};
    bp_shape_from_axes_sq(R, y0, nullptr, Q, nullptr);
  }
  double det = 100.0, det_old = 1.0;                          // :200-201
  int k = 0, status = BP_OK, rows_peak = 0, m_cur = 6;
  if (tid < 6) {                                              // init_halfspaces (:377-398)
    const int ax = tid >> 1;
    const double sgn = (tid & 1) ? -1.0 : 1.0;
    sA[3 * tid + 0] = ax == 0 ? sgn : 0.0;
    sA[3 * tid + 1] = ax == 1 ? sgn : 0.0;
    sA[3 * tid + 2] = ax == 2 ? sgn : 0.0;
    sb[tid] = pr.ws_rows[tid];
  }
  while (fabs(det - det_old) / det_old > 0.01) {              // :203
    ++k;
    if (k > pr.max_iter) break;                               // :204-207
    PassMetric pm;
    pass_metric_init(Q, &pm);
    __syncthreads();                                          // previous rows / control words consumed
    int st;
    {
      BP_PROF_T0();
      poly_pass<POLY, AW>(sc, sc_all.n, pm, p, s_dist, pr.cache_y, red_val, red_idx, sA, sb, pr.m_max, &m_cur, &st);
      BP_PROF_ADD(0);
    }
    rows_peak = m_cur > rows_peak ? m_cur : rows_peak;
    if (st == BP_OK && m_cur > pr.m_max) st = BP_ROW_OVERFLOW;
    if (st == BP_OK && (MODE == 1 || pr.optimize) && pr.row_cap > 0 && m_cur > pr.row_cap) st = BP_ROW_CAP;
    if (st != BP_OK) { status = st; break; }
    if (MODE == 0 && !pr.optimize) break;                     // :214-215
    if (MODE == 1) {
      __syncthreads();                                        // thread 0 has written the picked rows
      if (!pr.optimize) {                                     // :278-282: one free-centre MVIE, then out
        if (tid < 32) {
          double L[6], d[3];
          const int ms = bp_mvie_warp<9>(sA, sb, m_cur, p, scratch, L, d, nullptr);
          if (tid == 0) {
            double E[9], Qn[9], dq;
            bp_shape_from_L(L, E, Qn, &dq);
#pragma unroll
            for (int q = 0; q < 9; ++q) c_Q[q] = Qn[q];
            c_p[0] = d[0]; c_p[1] = d[1]; c_p[2] = d[2];
            c_status = ms;
          }
        }
      } else {
        det_old = det;                                        // :284
        if (tid < 32) {
          SharedRows rows{sA, sb};
          BpWarpRed red;
          double x[3];
          const int ms = bp_mvie_fixed_r(rows, m_cur, p, R, a_lb, red, x, nullptr);
          if (tid == 0) {
            double Qn[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, dq = 0.0;
            if (ms == BP_OK) bp_shape_from_axes(R, x, nullptr, Qn, &dq);
#pragma unroll
            for (int q = 0; q < 9; ++q) c_Q[q] = Qn[q];
            c_p[0] = p[0]; c_p[1] = p[1]; c_p[2] = p[2];
            c_det = dq;                                       // :299
            c_status = ms;
            c_small = (ms == BP_OK && fmin(x[0], fmin(x[1], x[2])) < 1e-3) ? 1 : 0;   // :293-294
          }
        }
      }
      __syncthreads();
      if (c_status != BP_OK) { status = c_status; break; }
#pragma unroll
      for (int q = 0; q < 9; ++q) Q[q] = c_Q[q];
      p[0] = c_p[0]; p[1] = c_p[1]; p[2] = c_p[2];
      if (!pr.optimize || c_small) break;                     // the small-axis exit leaves det alone (:293-299)
      det = c_det;
      continue;
    }
    det_old = det;                                            // :217
    // The trailing free-centre solve (:235-238) depends only on the rows of the pass the loop ends with and on the
    // seed.  It runs SPECULATIVELY on a second warp next to every pass's fixed-centre solve (the two solver warps
    // sit on different SM sub-partitions): if the loop ends with this pass the answer is (nearly) there, if the loop
    // goes on the primary warp raises c_abort and the speculative solve stops at its next Newton iteration.  Pass
    // max_iter is the last one whatever its MVIE returns (:204-207): no abort there.  BPGEO_SPEC=0 (pr.spec = 0)
    // speculates on that last pass only.
    const bool spec_final = MODE == 0 && pr.fixed_mid && k == pr.max_iter;
    const bool spec_any = MODE == 0 && pr.fixed_mid && pr.optimize && (spec_final || (SPEC && pr.spec));
    if (tid == 0) { c_abort = 0; f_done = 0; }
    __syncthreads();                                          // the picked rows are in shared memory
    if (warp_id == mw) {
      double L[6], d[3];
      BP_PROF_T0();
      const int ms = pr.fixed_mid ? bp_mvie_warp<6>(sA, sb, m_cur, p, scratch, L, d, nullptr)
                                  : bp_mvie_warp<9>(sA, sb, m_cur, p, scratch, L, d, nullptr);
      BP_PROF_ADD(1);
      if ((tid & 31) == 0) {
        double E[9], Qn[9], dq;
        bp_shape_from_L(L, E, Qn, &dq);
#pragma unroll
        for (int q = 0; q < 9; ++q) c_Q[q] = Qn[q];
        c_p[0] = d[0]; c_p[1] = d[1]; c_p[2] = d[2];
        c_det = dq;                                           // :229
        c_status = ms;
        const int small = (ms == BP_OK && bp_sym3_min_eig(E) < 1e-3) ? 1 : 0;   // :232-233
        c_small = small;
        // will the loop go on after this pass (:203-207, :232-233)?  Then (or on an error) nobody needs the
        // speculative trailing solve: stop it
        const bool goes_on = ms == BP_OK && !small && k < pr.max_iter && fabs(dq - det_old) / det_old > 0.01;
        if (spec_any && !spec_final && (goes_on || ms != BP_OK)) c_abort = 1;
      }
    } else if (spec_any && warp_id == mw2) {
      double L[6], d[3];
      BP_PROF_T0();
      int ms;
      if (SPEC && !spec_final) ms = bp_mvie_warp<9>(sA, sb, m_cur, p, scratch2, L, d, nullptr, &c_abort);
      else ms = bp_mvie_warp<9>(sA, sb, m_cur, p, scratch2, L, d, nullptr);
      BP_PROF_ADD(2);
      if ((tid & 31) == 0 && ms != BP_MVIE_ABORTED) {
        double E[9], Qn[9], dq;
        bp_shape_from_L(L, E, Qn, &dq);
#pragma unroll
        for (int q = 0; q < 9; ++q) f_Q[q] = Qn[q];
        f_p[0] = d[0]; f_p[1] = d[1]; f_p[2] = d[2];
        f_status = ms;
        f_done = 1;
      }
    }
    __syncthreads();
    have_final = f_done != 0;
    if (c_status != BP_OK) { status = c_status; break; }
#pragma unroll
    for (int q = 0; q < 9; ++q) Q[q] = c_Q[q];
    p[0] = c_p[0]; p[1] = c_p[1]; p[2] = c_p[2];
    det = c_det;
    if (c_small) break;
  }
  if (MODE == 0 && pr.optimize && pr.fixed_mid && status == BP_OK) {       // :235-238
    __syncthreads();
    if (!have_final && warp_id == mw) {
      double L[6], d[3];
      BP_PROF_T0();
      const int ms = bp_mvie_warp<9>(sA, sb, m_cur, p, scratch, L, d, nullptr);
      BP_PROF_ADD(2);
      if ((tid & 31) == 0) {
        double E[9], Qn[9], dq;
        bp_shape_from_L(L, E, Qn, &dq);
#pragma unroll
        for (int q = 0; q < 9; ++q) f_Q[q] = Qn[q];
        f_p[0] = d[0]; f_p[1] = d[1]; f_p[2] = d[2];
        f_status = ms;
      }
    }
    __syncthreads();
    if (f_status != BP_OK) status = f_status;
    else {
#pragma unroll
      for (int q = 0; q < 9; ++q) Q[q] = f_Q[q];
      p[0] = f_p[0]; p[1] = f_p[1]; p[2] = f_p[2];
    }
  }
  __syncthreads();
  // outputs: rows padded like normalize_set_size (A = 0, b = 10)
  const int m_out = m_cur < pr.m_max ? m_cur : pr.m_max;
  double* Arow = pr.A + (size_t)s * pr.m_max * 3;
  double* brow = pr.b + (size_t)s * pr.m_max;
  for (int r = tid; r < pr.m_max; r += blockDim.x) {
    const bool live = r < m_out;
    Arow[3 * r] = live ? sA[3 * r] : 0.0;
    Arow[3 * r + 1] = live ? sA[3 * r + 1] : 0.0;
    Arow[3 * r + 2] = live ? sA[3 * r + 2] : 0.0;
    brow[r] = live ? sb[r] : 10.0;
  }
  if (tid == 0) {
    pr.m[s] = m_out;
#pragma unroll
    for (int q = 0; q < 9; ++q) pr.q_ellipse[(size_t)s * 9 + q] = Q[q];
    pr.p_mid[3 * (size_t)s] = p[0]; pr.p_mid[3 * (size_t)s + 1] = p[1]; pr.p_mid[3 * (size_t)s + 2] = p[2];
    pr.status[s] = status;
    if (pr.iters) pr.iters[s] = k;
    if (pr.rows_peak) pr.rows_peak[s] = rows_peak;
  }
  if (MODE == 0 && (pr.aabb || pr.peers.world > 0 || pr.tail.S > 0)) {
    // Epilogue: the set's exact bounding box (the pair filter's input) while its rows are still in shared memory,
    // and -- multi-GPU -- the owner's stores of rows, row count and box straight into every rank's global tables
    // over NVLink: no separate box / scatter kernels, and a finished seed's stores overlap the seeds still running.
    __shared__ double e_red[4][6], e_box[6];
    for (int r = m_out + tid; r < pr.m_max; r += blockDim.x) {          // padding, as written to A / b above
      sA[3 * r] = 0.0; sA[3 * r + 1] = 0.0; sA[3 * r + 2] = 0.0; sb[r] = 10.0;
    }
    __syncthreads();
    cta_set_aabb(sA, sb, m_out, e_red, e_box);
    __syncthreads();
    if (pr.aabb && tid < 6) pr.aabb[(size_t)s * 6 + tid] = e_box[tid];
    const int g = pr.peers.slot0 + s;
    for (int r = 0; r < pr.peers.world; ++r) {
      char* base = (char*)pr.peers.base[r];
      double* Ad = (double*)(base + pr.peers.off_A) + (size_t)g * pr.m_max * 3;
      double* bd = (double*)(base + pr.peers.off_b) + (size_t)g * pr.m_max;
      for (int e = tid; e < 3 * pr.m_max; e += blockDim.x) Ad[e] = sA[e];
      for (int e = tid; e < pr.m_max; e += blockDim.x) bd[e] = sb[e];
      if (tid < 6) ((double*)(base + pr.peers.off_aabb))[(size_t)g * 6 + tid] = e_box[tid];
      if (tid == 6) ((int*)(base + pr.peers.off_m))[g] = m_out;
    }
    if (pr.tail.S > 0) {
      __syncthreads();                    // shared-memory rows are no longer needed: the dynamic area becomes scratch
      fused_tail_pairs(pr.tail, pr.peers, g, pr.m_max, e_box, s_dist);
    }
  }
#ifdef BPGEO_PROFILE
  if (tid == 0 && blockIdx.x < 65536) g_prof[4 * blockIdx.x + 3] = clock64() - prof_k0_;
#endif
}

// ---------------------------------------------------------------------------
// K3': greedy loop of find_set_collision_avoidance (ConvexSetFinder.py:309-375)
// ---------------------------------------------------------------------------
struct LineParams {
  const double* p0;          // [S,3]
  const double* p1;          // [S,3]
  double ws_rows[6];
  int limit_space;
  double e_max;
  double* A;
  double* b;
  int* m;
  int* status;
  int* collision;
  int m_max;
  int cache_x;               // polytope scenes: closest points kept in shared memory (x[3][N] | p_closest[3][N])
};

__device__ __forceinline__ double seg_closest(const double* p0, const double* d, const double* lb,
                                              const double* ub, double* x, double* pc) {
  double l2[3], u2[3], d2;
#pragma unroll
  for (int k = 0; k < 3; ++k) { l2[k] = lb[k] + 0.001; u2[k] = ub[k] - 0.001; }     // b - 0.001 (:496)
  double phi = bp_seg_box(p0, d, l2, u2, x, &d2);
#pragma unroll
  for (int k = 0; k < 3; ++k) pc[k] = p0[k] + phi * d[k];                             // :326
  double e0 = x[0] - pc[0], e1 = x[1] - pc[1], e2 = x[2] - pc[2];
  return sqrt(e0 * e0 + e1 * e1 + e2 * e2);                                           // :327
}

__global__ void __launch_bounds__(512) k_poly_line(SceneView sc_all, LineParams pr) {
  const SceneView sc = scene_of_item(sc_all, blockIdx.x);
  extern __shared__ double s_dist[];
  __shared__ double red_val[2][32];
  __shared__ int red_idx[2][32];
  const int s = blockIdx.x;
  const int tid = threadIdx.x, T = blockDim.x;
  double p0[3], p1[3], d[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    p0[k] = pr.p0[(size_t)s * 3 + k];
    p1[k] = pr.p1[(size_t)s * 3 + k];
    d[k] = p1[k] - p0[k];
  }
  double* Arow = pr.A + (size_t)s * pr.m_max * 3;
  double* brow = pr.b + (size_t)s * pr.m_max;
  if (tid < 6) {
    int ax = tid >> 1;
    double sgn = (tid & 1) ? -1.0 : 1.0;
    Arow[3 * tid + 0] = ax == 0 ? sgn : 0.0;
    Arow[3 * tid + 1] = ax == 1 ? sgn : 0.0;
    Arow[3 * tid + 2] = ax == 2 ? sgn : 0.0;
    // init_halfspaces_point: b = p[i] + e_max / -p[i] + e_max (:400-421)
    brow[tid] = pr.limit_space ? (sgn * p0[ax] + pr.e_max) : pr.ws_rows[tid];
  }
  double lmin = BP_INF;
  int lidx = 0x7fffffff;
  for (int j = tid; j < sc.n; j += T) {
    double lb[3], ub[3], x[3], pc[3];
    load_box(sc, j, lb, ub);
    double dd = seg_closest(p0, d, lb, ub, x, pc);
    s_dist[j] = dd;
    if (dd < lmin) { lmin = dd; lidx = j; }
  }
  int m_cur = 6, buf = 0, collision = 0;
  while (true) {
    double val = lmin;
    int idx = lidx;
    block_argmin(val, idx, red_val, red_idx, buf);
    if (!(val < BP_INF)) break;
    double lb[3], ub[3], x[3], pc[3];
    load_box(sc, idx, lb, ub);
    seg_closest(p0, d, lb, ub, x, pc);
    double a[3] = {x[0] - pc[0], x[1] - pc[1], x[2] - pc[2]};
    double nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    if (nrm < 1e-6) {                                  // line touches an obstacle (:336-345)
      collision = 1;
      a[0] = x[0] - p0[0]; a[1] = x[1] - p0[1]; a[2] = x[2] - p0[2];
      nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
      if (nrm < 1e-6) {
        a[0] = d[0]; a[1] = d[1]; a[2] = d[2];
        nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
      }
    }
    a[0] /= nrm; a[1] /= nrm; a[2] /= nrm;
    double bh = (a[0] * x[0] + a[1] * x[1] + a[2] * x[2]) - 0.001;    // :347
    if (tid == 0 && m_cur < pr.m_max) {
      Arow[3 * m_cur + 0] = a[0]; Arow[3 * m_cur + 1] = a[1]; Arow[3 * m_cur + 2] = a[2];
      brow[m_cur] = bh;
    }
    ++m_cur;
    lmin = BP_INF;
    lidx = 0x7fffffff;
    for (int j = tid; j < sc.n; j += T) {
      double dd = s_dist[j];
      if (!(dd < BP_INF)) continue;
      double l2[3], u2[3];
      load_box(sc, j, l2, u2);
      if (j == idx || bp_box_min_halfspace(a, bh, l2, u2) >= -1e-4) {   // unshrunk vertices (:352-357)
        s_dist[j] = BP_INF;
      } else if (dd < lmin) {
        lmin = dd; lidx = j;
      }
    }
  }
  for (int r = m_cur + tid; r < pr.m_max; r += T) {
    Arow[3 * r] = 0.0; Arow[3 * r + 1] = 0.0; Arow[3 * r + 2] = 0.0;
    brow[r] = 10.0;
  }
  if (tid == 0) {
    pr.m[s] = m_cur < pr.m_max ? m_cur : pr.m_max;
    pr.status[s] = m_cur > pr.m_max ? BP_ROW_OVERFLOW : BP_OK;
    pr.collision[s] = collision;
  }
}

// ---------------------------------------------------------------------------
// K3'p: find_set_collision_avoidance (:309-375) over GENERAL polytope obstacles.  Same greedy loop as k_poly_line;
// the closest points come from the segment-polytope QP (bp_seg_polytope_candidate), solved lazily like the point
// pass: the table starts with the distance from the segment to every obstacle's BOUNDING BOX (a lower bound),
// and only entries that can still win are refined, each by one warp (candidates dealt to the lanes).
// Dynamic shared memory: dist[N] | x[3][N] | p_closest[3][N].
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool seg_polytope_qp_warp(const double* rows4, int R, double shrink, const double* p0,
                                                     const double* d, double* x, double* phi_out, double* dist2) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  SmemRows4 rows{rows4};
  double best = BP_INF, bphi = BP_INF, xb[3] = {0.0, 0.0, 0.0}, xc[3], pc, oc;
  int bidx = 0x7fffffff, cnt = 0;
#define BP_SEGP_TRYW(I, J, K)                                                                                   \
  for (int pm = 0; pm < 3; ++pm) {                                                                              \
    if ((cnt & 31) == lane && bp_seg_polytope_candidate(rows, R, shrink, p0, d, (I), (J), (K), pm, xc, &pc, &oc) && \
        (bidx == 0x7fffffff || bp_seg_better(oc, pc, best, bphi))) {                                            \
      best = oc; bphi = pc; bidx = cnt; xb[0] = xc[0]; xb[1] = xc[1]; xb[2] = xc[2];                            \
    }                                                                                                           \
    ++cnt;                                                                                                      \
  }
  BP_SEGP_TRYW(-1, -1, -1)
  for (int i = 0; i < R; ++i) BP_SEGP_TRYW(i, -1, -1)
  for (int i = 0; i < R; ++i)
    for (int j = i + 1; j < R; ++j) BP_SEGP_TRYW(i, j, -1)
  for (int i = 0; i < R; ++i)
    for (int j = i + 1; j < R; ++j)
      for (int k = j + 1; k < R; ++k) BP_SEGP_TRYW(i, j, k)
#undef BP_SEGP_TRYW
  const double bmin = warp_min_nonneg(best);
  if (!(bmin < BP_INF)) return false;
  // least distance (to rounding), then the smallest phi (quirk Q9), then the first candidate
  const bool near = best <= bmin * (1.0 + 1e-12) + 1e-24;
  const double pmin = warp_min_nonneg(near ? (bphi < 0.0 ? 0.0 : bphi) : BP_INF);
  const unsigned cand = (near && bphi <= pmin) ? (unsigned)bidx : 0xffffffffu;
  const unsigned widx = __reduce_min_sync(full, cand);
  const int src = __ffs(__ballot_sync(full, cand == widx)) - 1;
  x[0] = __shfl_sync(full, xb[0], src);
  x[1] = __shfl_sync(full, xb[1], src);
  x[2] = __shfl_sync(full, xb[2], src);
  *phi_out = __shfl_sync(full, bphi, src);
  *dist2 = __shfl_sync(full, best, src);
  return true;
}

__global__ void __launch_bounds__(512) k_poly_line_p(SceneView sc_all, LineParams pr) {
  const SceneView sc = scene_of_item(sc_all, blockIdx.x);
  const int cache_x = pr.cache_x, n_tab = sc_all.n;     // n_tab: the table stride (largest scene of a batch)
  extern __shared__ double s_dist[];
  __shared__ double red_val[2][32];
  __shared__ int red_idx[2][32];
  __shared__ int s_list[BP_POLY_LIST];
  __shared__ int s_nlist;
  __shared__ double s_prow[16][BP_OBS_ROWS * 4];
  const int s = blockIdx.x;
  const int tid = threadIdx.x, T = blockDim.x;
  double* s_x = s_dist + n_tab;                // [3][N] when cache_x
  double* s_pc = s_dist + 4 * (size_t)n_tab;   // [3][N] when cache_x
  __shared__ double s_win[6];
  double p0[3], d[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    p0[k] = pr.p0[(size_t)s * 3 + k];
    d[k] = pr.p1[(size_t)s * 3 + k] - p0[k];
  }
  double* Arow = pr.A + (size_t)s * pr.m_max * 3;
  double* brow = pr.b + (size_t)s * pr.m_max;
  if (tid < 6) {
    int ax = tid >> 1;
    double sgn = (tid & 1) ? -1.0 : 1.0;
    Arow[3 * tid + 0] = ax == 0 ? sgn : 0.0;
    Arow[3 * tid + 1] = ax == 1 ? sgn : 0.0;
    Arow[3 * tid + 2] = ax == 2 ? sgn : 0.0;
    brow[tid] = pr.limit_space ? (sgn * p0[ax] + pr.e_max) : pr.ws_rows[tid];
  }
  if (tid == 0) s_nlist = 0;
  unsigned long long alive = 0ull;
  double lkey = BP_INF;
  int lidx = 0x3fffffff, lexact = 0;
  {
    int k = 0;
    for (int j = tid; j < sc.n; j += T, ++k) {
      double lb[3], ub[3], xb[3], d2;
      load_box(sc, j, lb, ub);
      bp_seg_box(p0, d, lb, ub, xb, &d2);                   // distance to the bounding box: a lower bound
      double bd = sqrt(d2) * (1.0 - 1e-9);
      if (!(bd > 0.0)) bd = DBL_MIN;
      s_dist[j] = -bd;
      alive |= 1ull << k;
      if (bd < lkey) { lkey = bd; lidx = j; }
    }
  }
  int m_cur = 6, buf = 0, collision = 0;
  while (true) {
    double val = lkey;
    int idx = lidx, exact = lexact;
    block_argmin_lazy(val, idx, exact, red_val, red_idx, buf);
    if (!(val < BP_INF)) break;
    if (!exact) {
      double lex = BP_INF;
      for (unsigned long long mk = alive; mk; mk &= mk - 1) {
        const double dv = s_dist[tid + (__ffsll((long long)mk) - 1) * T];
        if (dv >= 0.0) lex = fmin(lex, dv);
      }
      const double ex = block_min_nonneg(lex, red_val, buf);
      const double thr = fmax(ex < BP_INF ? ex : 0.0, BP_LAZY_GROW * val);
      for (unsigned long long mk = alive; mk; mk &= mk - 1) {
        const int j = tid + (__ffsll((long long)mk) - 1) * T;
        const double dv = s_dist[j];
        if (dv < 0.0 && -dv <= thr) {
          const int slot = atomicAdd(&s_nlist, 1);
          if (slot < BP_POLY_LIST) s_list[slot] = j;
        }
      }
      __syncthreads();
      const int nl = s_nlist < BP_POLY_LIST ? s_nlist : BP_POLY_LIST;
      const int warp = tid >> 5, lane = tid & 31, nw = T >> 5;
      for (int q = warp; q < nl; q += nw) {
        const int j = s_list[q];
        const int R = sc.nrows[j];
        for (int e = lane; e < R * 4; e += 32) s_prow[warp][e] = __ldg(sc.rows + (size_t)j * BP_OBS_ROWS * 4 + e);
        __syncwarp();
        double x[3], phi, d2;
        const bool okq = seg_polytope_qp_warp(s_prow[warp], R, 0.001, p0, d, x, &phi, &d2);   // b - 0.001 (:496)
        if (lane == 0) {
          s_dist[j] = okq ? sqrt(d2) : BP_INF;               // :327
          if (cache_x) {
            s_x[j] = x[0]; s_x[n_tab + j] = x[1]; s_x[2 * n_tab + j] = x[2];
            s_pc[j] = p0[0] + phi * d[0]; s_pc[n_tab + j] = p0[1] + phi * d[1]; s_pc[2 * n_tab + j] = p0[2] + phi * d[2];
          }
        }
        __syncwarp();
      }
      __syncthreads();
      if (tid == 0) s_nlist = 0;
      lkey = BP_INF; lidx = 0x3fffffff; lexact = 0;
      for (unsigned long long mk = alive; mk; mk &= mk - 1) {
        const int kk = __ffsll((long long)mk) - 1;
        const int j = tid + kk * T;
        double dv = s_dist[j];
        if (!(dv < BP_INF)) { alive &= ~(1ull << kk); continue; }     // empty polytope
        const int e = dv >= 0.0;
        dv = fabs(dv);
        if (dv < lkey || (dv == lkey && e < lexact)) { lkey = dv; lidx = j; lexact = e; }
      }
      continue;
    }
    double x[3], pc[3];
    if (cache_x) {
      x[0] = s_x[idx]; x[1] = s_x[n_tab + idx]; x[2] = s_x[2 * n_tab + idx];
      pc[0] = s_pc[idx]; pc[1] = s_pc[n_tab + idx]; pc[2] = s_pc[2 * n_tab + idx];
    } else {                                     // large scenes: warp 0 re-solves the winner's QP (same bits)
      if (tid < 32) {
        const int R = sc.nrows[idx];
        for (int e = tid; e < R * 4; e += 32) s_prow[0][e] = __ldg(sc.rows + (size_t)idx * BP_OBS_ROWS * 4 + e);
        __syncwarp();
        double xw[3] = {0.0, 0.0, 0.0}, phiw = 0.0, d2w = 0.0;
        seg_polytope_qp_warp(s_prow[0], R, 0.001, p0, d, xw, &phiw, &d2w);
        if (tid == 0) {
          s_win[0] = xw[0]; s_win[1] = xw[1]; s_win[2] = xw[2];
          s_win[3] = p0[0] + phiw * d[0]; s_win[4] = p0[1] + phiw * d[1]; s_win[5] = p0[2] + phiw * d[2];
        }
      }
      __syncthreads();
      x[0] = s_win[0]; x[1] = s_win[1]; x[2] = s_win[2]; pc[0] = s_win[3]; pc[1] = s_win[4]; pc[2] = s_win[5];
      __syncthreads();
    }
    double a[3] = {x[0] - pc[0], x[1] - pc[1], x[2] - pc[2]};
    double nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    if (nrm < 1e-6) {                                  // line touches an obstacle (:336-345)
      collision = 1;
      a[0] = x[0] - p0[0]; a[1] = x[1] - p0[1]; a[2] = x[2] - p0[2];
      nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
      if (nrm < 1e-6) {
        a[0] = d[0]; a[1] = d[1]; a[2] = d[2];
        nrm = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
      }
    }
    a[0] /= nrm; a[1] /= nrm; a[2] /= nrm;
    double bh = (a[0] * x[0] + a[1] * x[1] + a[2] * x[2]) - 0.001;    // :347
    if (tid == 0 && m_cur < pr.m_max) {
      Arow[3 * m_cur + 0] = a[0]; Arow[3 * m_cur + 1] = a[1]; Arow[3 * m_cur + 2] = a[2];
      brow[m_cur] = bh;
    }
    ++m_cur;
    lkey = BP_INF; lidx = 0x3fffffff; lexact = 0;
    for (unsigned long long mk = alive; mk; mk &= mk - 1) {
      const int kk = __ffsll((long long)mk) - 1;
      const int j = tid + kk * T;
      if (j == idx || poly_min_halfspace(sc, j, a, bh) >= -1e-4) {   // unshrunk vertices (:352-357)
        alive &= ~(1ull << kk);
      } else {
        double dv = s_dist[j];
        const int e = dv >= 0.0;
        dv = fabs(dv);
        if (dv < lkey || (dv == lkey && e < lexact)) { lkey = dv; lidx = j; lexact = e; }
      }
    }
  }
  for (int r = m_cur + tid; r < pr.m_max; r += T) {
    Arow[3 * r] = 0.0; Arow[3 * r + 1] = 0.0; Arow[3 * r + 2] = 0.0;
    brow[r] = 10.0;
  }
  if (tid == 0) {
    pr.m[s] = m_cur < pr.m_max ? m_cur : pr.m_max;
    pr.status[s] = m_cur > pr.m_max ? BP_ROW_OVERFLOW : BP_OK;
    pr.collision[s] = collision;
  }
}

// ---------------------------------------------------------------------------
// K4: MVIE, one warp (one 32-thread CTA) per set -- see bp_mvie_warp.cuh.
// mode 0: loop step with fixed centre   (mvie_socp_fixed_mid, :220-221)
// mode 1: loop step with free centre    (mvie_socp, :222-223)
// mode 2: final free-centre solve after the loop (:235-238), no loop control
// mode 3: standalone (bp_mvie), centre/hint from `centre`, free_centre flag
// ---------------------------------------------------------------------------
struct MvieParams {
  const double* A;
  const double* b;
  const int* m;
  int S;
  int m_max;
  int mode;
  int free_centre;            // mode 3
  SeedState* state;           // modes 0-2
  const double* centre;       // mode 3 [S,3]
  const double* hint;         // mode 2 optional [S,3] hint (line sets: p0)
  double* q_inv_out;          // mode 3
  double* q_ellipse_out;      // mode 3, and export target of modes 0-2 when non-null
  double* centre_out;
  int* status_out;
  int* iters_out;             // newton iterations (mode 3) or NULL
};

__global__ void __launch_bounds__(32) k_mvie(MvieParams pr) {
  __shared__ double scratch[BP_MVIE_SCRATCH_DOUBLES];
  const int lane = threadIdx.x;
  const int s = blockIdx.x;                 // one warp (= one CTA) per set: everything below is warp-uniform
  SeedState* st = nullptr;
  double c0[3];
  if (pr.mode <= 2) {
    st = pr.state + s;
    const bool run = (st->status == BP_OK) && (pr.mode == 2 || st->active);
    if (!run) return;
    c0[0] = st->p[0]; c0[1] = st->p[1]; c0[2] = st->p[2];
    if (pr.mode == 2 && pr.hint) { c0[0] = pr.hint[3 * s]; c0[1] = pr.hint[3 * s + 1]; c0[2] = pr.hint[3 * s + 2]; }
  } else {
    c0[0] = pr.centre[3 * s]; c0[1] = pr.centre[3 * s + 1]; c0[2] = pr.centre[3 * s + 2];
  }
  const int m = pr.m[s];
  const double* A = pr.A + (size_t)s * pr.m_max * 3;
  const double* b = pr.b + (size_t)s * pr.m_max;
  double L[6], d[3];
  int iters = 0;
  const bool free_c = (pr.mode == 1 || pr.mode == 2 || (pr.mode == 3 && pr.free_centre));
  int status = free_c ? bp_mvie_warp<9>(A, b, m, c0, scratch, L, d, &iters)
                      : bp_mvie_warp<6>(A, b, m, c0, scratch, L, d, &iters);
  if (status == BP_MVIE_NO_INTERIOR && free_c) {
    // the hint is not strictly inside (e.g. mvie_socp called without one): find an
    // interior point with the phase-I LP of K6 on the set's own rows, then retry
    __syncwarp();
    double xi[3];
    if (bp_pair_feasible_warp(A, b, m, A, b, 0, 1e-9, scratch, nullptr, xi)) {
      __syncwarp();
      status = bp_mvie_warp<9>(A, b, m, xi, scratch, L, d, &iters);
    }
  }
  if (lane != 0) return;
  double E[9], Q[9], detQ;
  bp_shape_from_L(L, E, Q, &detQ);
  if (pr.mode <= 2) {
    if (status != BP_OK) { st->status = status; st->active = 0; return; }
    if (pr.mode < 2) st->det_old = st->det;             // :217
#pragma unroll
    for (int k = 0; k < 9; ++k) st->Q[k] = Q[k];
    st->p[0] = d[0]; st->p[1] = d[1]; st->p[2] = d[2];
    if (pr.mode < 2) {
      st->det = detQ;                                    // :229
      if (bp_sym3_min_eig(E) < 1e-3) st->active = 0;     // :232-233
    }
  } else {
#pragma unroll
    for (int k = 0; k < 9; ++k) { pr.q_inv_out[(size_t)s * 9 + k] = E[k]; pr.q_ellipse_out[(size_t)s * 9 + k] = Q[k]; }
    pr.centre_out[3 * s] = d[0]; pr.centre_out[3 * s + 1] = d[1]; pr.centre_out[3 * s + 2] = d[2];
    pr.status_out[s] = status;
    if (pr.iters_out) pr.iters_out[s] = iters;
  }
}

// K4b: one warp per set (mvie_socp_fixed_r, :564-588)
__global__ void __launch_bounds__(32) k_mvie_fixed_r(const double* __restrict__ A, const double* __restrict__ b,
                                                     const int* __restrict__ m, int m_max,
                                                     const double* __restrict__ centre, const double* __restrict__ Rs,
                                                     const double* __restrict__ a_lb, double* __restrict__ q_inv_out,
                                                     double* __restrict__ q_ellipse_out, double* __restrict__ eigs_out,
                                                     int* __restrict__ status_out, int* __restrict__ iters_out) {
  const int s = blockIdx.x;
  GlobalRows rows{A + (size_t)s * m_max * 3, b + (size_t)s * m_max};
  BpWarpRed red;
  double p[3], R[9], x[3] = {0.0, 0.0, 0.0};
#pragma unroll
  for (int k = 0; k < 3; ++k) p[k] = centre[3 * (size_t)s + k];
#pragma unroll
  for (int k = 0; k < 9; ++k) R[k] = Rs[9 * (size_t)s + k];
  int iters = 0;
  const int st = bp_mvie_fixed_r(rows, m[s], p, R, a_lb[s], red, x, &iters);
  if (threadIdx.x != 0) return;
  double E[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, Q[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  if (st == BP_OK) bp_shape_from_axes(R, x, E, Q, nullptr);
#pragma unroll
  for (int k = 0; k < 9; ++k) { q_inv_out[9 * (size_t)s + k] = E[k]; q_ellipse_out[9 * (size_t)s + k] = Q[k]; }
#pragma unroll
  for (int k = 0; k < 3; ++k) eigs_out[3 * (size_t)s + k] = x[k];
  status_out[s] = st;
  if (iters_out) iters_out[s] = iters;
}

__global__ void k_state_init(SeedState* st, const double* __restrict__ seeds, int S) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  SeedState v;
#pragma unroll
  for (int k = 0; k < 9; ++k) v.Q[k] = 0.0;
  v.Q[0] = v.Q[4] = v.Q[8] = 1.0 / 1e-4;                 // q_ellipse = diag(1/a) (:192-194)
  v.p[0] = seeds[3 * s]; v.p[1] = seeds[3 * s + 1]; v.p[2] = seeds[3 * s + 2];
  v.det = 100.0; v.det_old = 1.0;                        // :200-201
  v.k = 0; v.active = 1; v.status = BP_OK; v.rows_peak = 0;
  st[s] = v;
}

__global__ void k_state_export(const SeedState* st, int S, int max_iter, double* __restrict__ q_ellipse,
                               double* __restrict__ p_mid, int* __restrict__ status, int* __restrict__ iters,
                               int* __restrict__ rows_peak) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  if (q_ellipse) {
#pragma unroll
    for (int k = 0; k < 9; ++k) q_ellipse[(size_t)s * 9 + k] = st[s].Q[k];
  }
  if (p_mid) { p_mid[3 * s] = st[s].p[0]; p_mid[3 * s + 1] = st[s].p[1]; p_mid[3 * s + 2] = st[s].p[2]; }
  if (status) status[s] = st[s].status;
  if (rows_peak) rows_peak[s] = st[s].rows_peak;
  if (iters) {
    // the reference's while test runs once more after the last pass and bumps k
    // before breaking on k > max_iter (:203-207)
    int k = st[s].k;
    if (st[s].active && st[s].status == BP_OK && k >= max_iter &&
        fabs(st[s].det - st[s].det_old) / st[s].det_old > 0.01) ++k;
    iters[s] = k;
  }
}

// line sets: seed the state for the trailing free-centre MVIE (:370-374)
__global__ void k_state_init_line(SeedState* st, const double* __restrict__ p0, const int* __restrict__ status, int S) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  SeedState v;
#pragma unroll
  for (int k = 0; k < 9; ++k) v.Q[k] = 0.0;
  v.p[0] = p0[3 * s]; v.p[1] = p0[3 * s + 1]; v.p[2] = p0[3 * s + 2];
  v.det = 100.0; v.det_old = 1.0;
  v.k = 0; v.active = 0; v.status = status[s]; v.rows_peak = 0;
  st[s] = v;
}

// ---------------------------------------------------------------------------
// K6: pairwise feasibility (BoundPlanner.set_intersection, BoundPlanner.py:774-798).
// Three kernels per call:
//   k_set_aabb      one CTA per set: exact axis-aligned bounding box of the
//                   polytope by vertex enumeration (all row triples);
//   k_pair_filter   every pair (i, j>i) of the row block: pairs whose boxes are
//                   disjoint cannot intersect (the tol-shrunk sets lie inside
//                   the unshrunk boxes) -> bit stays 0; the others are appended
//                   to a compact work list (warp-aggregated atomics);
//   k_pair_lp       persistent grid over the work list, one WARP per surviving
//                   pair (bp_lp_warp.cuh: rows across lanes, warp-uniform
//                   phase-I Newton), result bits set with atomicOr.
// The filter only decides WHO runs the LP; every answer that is 1 comes from
// the LP, every 0 from the LP or from a rigorous box separation.
// ---------------------------------------------------------------------------

#define BP_LP_T0_SCALE 8.0

__global__ void __launch_bounds__(128) k_set_aabb(const double* __restrict__ A, const double* __restrict__ b,
                                                  const int* __restrict__ m, int S, int m_max,
                                                  double* __restrict__ aabb) {
  __shared__ double red[4][6];
  const int s = blockIdx.x;                     // one 128-thread CTA per set
  cta_set_aabb(A + (size_t)s * m_max * 3, b + (size_t)s * m_max, m[s], red, aabb + (size_t)s * 6);
}

// Block = 8 rows i x 32 columns j.
__global__ void __launch_bounds__(256) k_pair_filter(const double* __restrict__ aabb, int S, int row_begin, int row_end,
                                                     int2* __restrict__ list, unsigned int* __restrict__ count) {
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  const int i = row_begin + blockIdx.y * 8 + wy;
  const int j = blockIdx.x * 32 + lane;
  if (i >= row_end) return;
  bool keep = false;
  if (j < S && j > i) {
    keep = true;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double loi = __ldg(aabb + (size_t)i * 6 + k), hii = __ldg(aabb + (size_t)i * 6 + 3 + k);
      const double loj = __ldg(aabb + (size_t)j * 6 + k), hij = __ldg(aabb + (size_t)j * 6 + 3 + k);
      if (loi > hij + BP_AABB_EPS || loj > hii + BP_AABB_EPS) keep = false;
    }
  }
  const unsigned int mask = __ballot_sync(0xffffffffu, keep);
  if (mask == 0) return;
  unsigned int base = 0;
  if (lane == 0) base = atomicAdd(count, __popc(mask));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (keep) list[base + __popc(mask & ((1u << lane) - 1u))] = make_int2(i, j);
}

// Rigorous pre-test of one pair by one warp, using the sets' bounding boxes AND the tolerance: a point x of the
// tol-shrunk set j (a_s.x <= b_s - tol for every row) has the ball B(x, rho_j), rho_j = tol / max_s |a_s|, inside
// the unshrunk set j, hence inside its bounding box: x lies in the box eroded by rho_j.  The pair is disjoint when
//   * the two eroded boxes do not overlap, or
//   * for some row r of set i the smallest a_r.x over the eroded box of j already exceeds b_r - tol
//     (the oriented test the box-box test misses), or the same with i and j exchanged.
// Only "disjoint" is ever concluded here; every "intersects" still comes from the LP.
template <bool G>
__device__ __forceinline__ double bp_ldv(const double* p) { return G ? __ldg(p) : *p; }
// G: the operands are read-only global memory (ld.global.nc); else plain loads (shared-memory staging of the tail)
template <bool G = true>
__device__ __forceinline__ bool bp_pair_margin_reject(const double* Ai, const double* bi, int mi, const double* boxi,
                                                      const double* Aj, const double* bj, int mj, const double* boxj,
                                                      double tol) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  double lo_i[3], hi_i[3], lo_j[3], hi_j[3];
  bool finite = true;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    lo_i[k] = bp_ldv<G>(boxi + k); hi_i[k] = bp_ldv<G>(boxi + 3 + k);
    lo_j[k] = bp_ldv<G>(boxj + k); hi_j[k] = bp_ldv<G>(boxj + 3 + k);
    finite = finite && fabs(lo_i[k]) < 1e6 && fabs(hi_i[k]) < 1e6 && fabs(lo_j[k]) < 1e6 && fabs(hi_j[k]) < 1e6;
  }
  if (!finite) return false;                       // no bounding box (unbounded / degenerate description)
  // largest row norm of each set
  double ni = 0.0, nj = 0.0;
  for (int r = lane; r < mi; r += 32) {
    const double a0 = bp_ldv<G>(Ai + 3 * r), a1 = bp_ldv<G>(Ai + 3 * r + 1), a2 = bp_ldv<G>(Ai + 3 * r + 2);
    ni = fmax(ni, a0 * a0 + a1 * a1 + a2 * a2);
  }
  for (int r = lane; r < mj; r += 32) {
    const double a0 = bp_ldv<G>(Aj + 3 * r), a1 = bp_ldv<G>(Aj + 3 * r + 1), a2 = bp_ldv<G>(Aj + 3 * r + 2);
    nj = fmax(nj, a0 * a0 + a1 * a1 + a2 * a2);
  }
  ni = sqrt(-bp_warp_min(-ni));
  nj = sqrt(-bp_warp_min(-nj));
  if (!(ni > 0.0) || !(nj > 0.0) || !(tol >= 0.0)) return false;
  // erosion, kept a hair smaller than rho so that rounding can only weaken the test
  const double ri = (tol / ni) * (1.0 - 1e-9) - BP_AABB_EPS, rj = (tol / nj) * (1.0 - 1e-9) - BP_AABB_EPS;
  bool apart = false;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    lo_i[k] += ri; hi_i[k] -= ri; lo_j[k] += rj; hi_j[k] -= rj;
    if (lo_i[k] > hi_i[k] || lo_j[k] > hi_j[k]) apart = true;            // a shrunk set is empty
    if (lo_i[k] > hi_j[k] || lo_j[k] > hi_i[k]) apart = true;            // eroded boxes apart
  }
  if (!apart) {
    for (int r = lane; r < mi; r += 32) {           // rows of i against the eroded box of j
      const double a0 = bp_ldv<G>(Ai + 3 * r), a1 = bp_ldv<G>(Ai + 3 * r + 1), a2 = bp_ldv<G>(Ai + 3 * r + 2);
      const double mu = (fmin(a0 * lo_j[0], a0 * hi_j[0]) + fmin(a1 * lo_j[1], a1 * hi_j[1])) + fmin(a2 * lo_j[2], a2 * hi_j[2]);
      const double rhs = bp_ldv<G>(bi + r) - tol;
      if (mu - rhs > 1e-9 * (1.0 + fabs(rhs))) apart = true;
    }
    for (int r = lane; r < mj; r += 32) {           // rows of j against the eroded box of i
      const double a0 = bp_ldv<G>(Aj + 3 * r), a1 = bp_ldv<G>(Aj + 3 * r + 1), a2 = bp_ldv<G>(Aj + 3 * r + 2);
      const double mu = (fmin(a0 * lo_i[0], a0 * hi_i[0]) + fmin(a1 * lo_i[1], a1 * hi_i[1])) + fmin(a2 * lo_i[2], a2 * hi_i[2]);
      const double rhs = bp_ldv<G>(bj + r) - tol;
      if (mu - rhs > 1e-9 * (1.0 + fabs(rhs))) apart = true;
    }
  }
  return __any_sync(full, apart);
}

// (122 registers: two CTAs per SM.  Holding the allocation to 80 registers for three CTAs per SM spills and was
// measured slower on both the 1.7 k LPs of C2 (0.064 vs 0.055 ms) and the ~10 k LPs of C4 (0.113 vs 0.109 ms).)
__global__ void __launch_bounds__(256) k_pair_lp(const double* __restrict__ A, const double* __restrict__ b,
                                                 const int* __restrict__ m, int S, int m_max, double tol,
                                                 int row_begin, const double* __restrict__ aabb,
                                                 const int2* __restrict__ list,
                                                 unsigned int* __restrict__ count,
                                                 unsigned int* __restrict__ adj, double* __restrict__ x_feas) {
  __shared__ double scratch[8][BP_LP_SCRATCH_DOUBLES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int words = (S + 31) >> 5;
  const unsigned int n = count[0];
  // One warp per surviving pair, taken from a shared cursor (count[1], zeroed with the list count): the grid holds
  // exactly the CTAs that are resident at once, and a warp that drew short LPs takes more of them.  (A strided
  // static split over a larger grid ran in waves, each paying the latency of its slowest LPs: 0.29 ms instead of
  // 0.1 ms for the 13.6 k LPs of a rank of the 8-GPU graph.)
  for (;;) {
    unsigned int p = 0;
    if (lane == 0) p = atomicAdd(count + 1, 1u);
    p = __shfl_sync(0xffffffffu, p, 0);
    if (p >= n) break;
    const int2 pr = list[p];
    if (bp_pair_margin_reject(A + (size_t)pr.x * m_max * 3, b + (size_t)pr.x * m_max, m[pr.x], aabb + (size_t)pr.x * 6,
                              A + (size_t)pr.y * m_max * 3, b + (size_t)pr.y * m_max, m[pr.y], aabb + (size_t)pr.y * 6,
                              tol)) {
#ifdef BPGEO_PROFILE
      if (lane == 0) atomicAdd((unsigned long long*)&g_prof_pair[68], 1ull);
#endif
      continue;
    }
    double xi[3], x0[3], region[6];
    bool have_region = true;
#pragma unroll
    for (int k = 0; k < 3; ++k) {                       // start at the middle of the overlap of the two boxes
      const double lo = fmax(__ldg(aabb + (size_t)pr.x * 6 + k), __ldg(aabb + (size_t)pr.y * 6 + k));
      const double hi = fmin(__ldg(aabb + (size_t)pr.x * 6 + 3 + k), __ldg(aabb + (size_t)pr.y * 6 + 3 + k));
      x0[k] = 0.5 * (lo + hi);
      if (!(fabs(x0[k]) < 1e6)) x0[k] = 0.0;            // unbounded description: no box
      region[k] = lo - BP_AABB_EPS; region[3 + k] = hi + BP_AABB_EPS;     // every common point lies in this box
      have_region = have_region && fabs(lo) < 1e6 && fabs(hi) < 1e6;
    }
    const double* reg = have_region ? region : nullptr;
#ifdef BPGEO_PROFILE
    int lp_iters = 0;
    const long long lp_t0 = clock64();
    const int res = bp_pair_feasible_warp(A + (size_t)pr.x * m_max * 3, b + (size_t)pr.x * m_max, m[pr.x],
                                          A + (size_t)pr.y * m_max * 3, b + (size_t)pr.y * m_max, m[pr.y], tol,
                                          scratch[wib], &lp_iters, xi, x0, BP_LP_T0_SCALE, reg);
    if (lane == 0) {
      int bk = lp_iters / 2; if (bk > 63) bk = 63;
      atomicAdd((unsigned long long*)&g_prof_pair[bk], 1ull);
      atomicAdd((unsigned long long*)&g_prof_pair[64], 1ull);
      atomicAdd((unsigned long long*)&g_prof_pair[65], (unsigned long long)lp_iters);
      atomicMax((unsigned long long*)&g_prof_pair[66], (unsigned long long)(clock64() - lp_t0));
      if (res) atomicAdd((unsigned long long*)&g_prof_pair[67], 1ull);
    }
#else
    const int res = bp_pair_feasible_warp(A + (size_t)pr.x * m_max * 3, b + (size_t)pr.x * m_max, m[pr.x],
                                          A + (size_t)pr.y * m_max * 3, b + (size_t)pr.y * m_max, m[pr.y], tol,
                                          scratch[wib], nullptr, xi, x0, BP_LP_T0_SCALE, reg);
#endif
    if (lane == 0 && res) {
      atomicOr(adj + (size_t)(pr.x - row_begin) * words + (pr.y >> 5), 1u << (pr.y & 31));
      if (x_feas) {
        double* xo = x_feas + ((size_t)(pr.x - row_begin) * S + pr.y) * 3;
        xo[0] = xi[0]; xo[1] = xi[1]; xo[2] = xi[2];
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Tail of the fused set build: pair tests by the CTAs whose set is finished (TailParams above).
// Every rank's tables hold an ARRIVAL LOG: a counter that grows by one per arrived set (S per step, never reset)
// and a ring of S entries (epoch, set id).  A CTA whose set is finished
//   1. snapshots the counter: the sets logged before are NOT its business -- their CTAs are waiting and will see
//      this set arrive (snapshot BEFORE publishing: of two sets each pair is then tested by at least one of them,
//      by both only when they finish within a memory round trip of each other; results are idempotent atomicOr's);
//   2. publishes: fence, then in every rank's log a slot (atomicAdd on the counter) and the entry (release);
//   3. follows its own rank's log from the snapshot on until all S sets of the step are there: an arriving set is
//      box-tested against this one (the k_pair_filter test), survivors go through the margin pre-test and the LP of
//      k_pair_lp, one warp per pair, on rows staged in shared memory with coherent loads; a 1 is OR-ed into row
//      min(g,h) of every rank's adjacency.  One polled word per waiting CTA, O(1) work per arrival.
// All CTAs of the launch must be resident at once (a waiting CTA never yields its SM): the host checks that.
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long bp_ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void bp_st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned int bp_ld_relaxed_sys_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __noinline__ void fused_tail_pairs(TailParams tp, PeerTables peers, int g, int m_max, const double* my_box,
                                              double* work) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ int t_list[128];
  __shared__ int t_n;
  __shared__ unsigned int t_cnt;
  const int epoch = *tp.epoch;
  const unsigned int S = (unsigned int)tp.S;
  const unsigned int base = (unsigned int)(epoch - 1) * S;        // counter value at the start of this step
  double bx[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) bx[k] = my_box[k];
  // 1. snapshot
  if (tid == 0) t_cnt = bp_ld_relaxed_sys_u32(tp.count) - base;
  __syncthreads();
  unsigned int seen = t_cnt;
  // 2. publish (the table stores of the epilogue first)
  __threadfence_system();
  __syncthreads();
  if (tid < (peers.world > 0 ? peers.world : 1)) {
    unsigned int* cnt = peers.world > 0 ? (unsigned int*)((char*)peers.base[tid] + tp.off_count) : tp.count;
    unsigned long long* lg = peers.world > 0 ? (unsigned long long*)((char*)peers.base[tid] + tp.off_log) : tp.log;
    const unsigned int slot = atomicAdd(cnt, 1u) - base;
    bp_st_release_sys_u64(lg + (slot % S), ((unsigned long long)(unsigned int)epoch << 32) | (unsigned int)g);
  }
  const size_t par_off = peers.world > 0 ? (size_t)(epoch & 1) * tp.S * tp.words : 0;
  constexpr int SET_D = BP_MAX_ROWS * 4 + 8;            // rows [48*3] | b [48] | box [6] (+2)
  double* lp_scr = work + warp * (BP_LP_SCRATCH_DOUBLES + 2 * SET_D);
  double* set_lo = lp_scr + BP_LP_SCRATCH_DOUBLES;
  double* set_hi = set_lo + SET_D;
  // 3. the sets that arrive from the snapshot on
  while (seen < S) {
    __syncthreads();                                   // t_cnt / t_list of the previous trip consumed
    if (tid == 0) { t_cnt = bp_ld_relaxed_sys_u32(tp.count) - base; t_n = 0; }
    __syncthreads();
    unsigned int n_new = t_cnt - seen;
    if (n_new == 0) { __nanosleep(400); continue; }
    if (n_new > 128) n_new = 128;
    if ((unsigned int)tid < n_new) {
      unsigned long long e;
      do {                                             // the entry follows its counter increment within a round trip
        e = bp_ld_acquire_sys_u64(tp.log + ((seen + tid) % S));
      } while ((int)(e >> 32) != epoch);
      const int h = (int)(unsigned int)e;
      if (h != g) {
        const volatile double* bh = tp.aabb + (size_t)h * 6;
        bool keep = true;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double loj = bh[k], hij = bh[3 + k];
          if (bx[k] > hij + BP_AABB_EPS || loj > bx[3 + k] + BP_AABB_EPS) keep = false;
        }
        if (keep) t_list[atomicAdd(&t_n, 1)] = h;
      }
    }
    __syncthreads();
    seen += n_new;
    const int n = t_n;
    for (int e = warp; e < n; e += 4) {
      const int h = t_list[e];
      const int lo = g < h ? g : h, hi = g < h ? h : g;
      const int mlo = *(const volatile int*)(tp.m + lo), mhi = *(const volatile int*)(tp.m + hi);
      const volatile double* Al = tp.A + (size_t)lo * m_max * 3;
      const volatile double* bl = tp.b + (size_t)lo * m_max;
      const volatile double* Ah = tp.A + (size_t)hi * m_max * 3;
      const volatile double* bhh = tp.b + (size_t)hi * m_max;
      for (int x = lane; x < mlo * 3; x += 32) set_lo[x] = Al[x];
      for (int x = lane; x < mlo; x += 32) set_lo[BP_MAX_ROWS * 3 + x] = bl[x];
      for (int x = lane; x < mhi * 3; x += 32) set_hi[x] = Ah[x];
      for (int x = lane; x < mhi; x += 32) set_hi[BP_MAX_ROWS * 3 + x] = bhh[x];
      if (lane < 6) {
        set_lo[BP_MAX_ROWS * 4 + lane] = ((const volatile double*)tp.aabb)[(size_t)lo * 6 + lane];
        set_hi[BP_MAX_ROWS * 4 + lane] = ((const volatile double*)tp.aabb)[(size_t)hi * 6 + lane];
      }
      __syncwarp();
      const double* boxl = set_lo + BP_MAX_ROWS * 4;
      const double* boxh = set_hi + BP_MAX_ROWS * 4;
      int res = 0;
      if (!bp_pair_margin_reject<false>(set_lo, set_lo + BP_MAX_ROWS * 3, mlo, boxl, set_hi, set_hi + BP_MAX_ROWS * 3, mhi,
                                        boxh, tp.tol)) {
        double xi[3], x0[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {                   // start at the middle of the overlap of the two boxes
          const double lov = fmax(boxl[k], boxh[k]);
          const double hiv = fmin(boxl[3 + k], boxh[3 + k]);
          x0[k] = 0.5 * (lov + hiv);
          if (!(fabs(x0[k]) < 1e6)) x0[k] = 0.0;
        }
        res = bp_pair_feasible_warp(set_lo, set_lo + BP_MAX_ROWS * 3, mlo, set_hi, set_hi + BP_MAX_ROWS * 3, mhi, tp.tol,
                                    lp_scr, nullptr, xi, x0, BP_LP_T0_SCALE);
      }
      if (lane == 0 && res) {
        const size_t word = par_off + (size_t)lo * tp.words + (hi >> 5);
        const unsigned int bit = 1u << (hi & 31);
        if (peers.world > 0) {
          for (int r = 0; r < peers.world; ++r)
            atomicOr((unsigned int*)((char*)peers.base[r] + tp.off_bits) + word, bit);
        } else {
          atomicOr(tp.bits + word, bit);
        }
      }
      __syncwarp();
    }
  }
}

// start of a step of the tail pipelines: next epoch; the adjacency buffer the NEXT step will use is cleared now
// (it was last written two steps ago, and nobody writes it before every rank has passed this step's final barrier)
__global__ void k_step_begin(const int* epoch, unsigned int* bits, size_t words_per_buffer, int double_buffered) {
  const int ep = *epoch + 1;                       // (the increment itself is k_step_epoch, launched after this)
  unsigned int* buf = bits + (double_buffered ? (size_t)((ep + 1) & 1) * words_per_buffer : 0);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < words_per_buffer; i += (size_t)gridDim.x * blockDim.x)
    buf[i] = 0u;
}
__global__ void k_step_epoch(int* epoch) { *epoch += 1; }

// K6 over an explicit pair list (batched planner rounds: the pairs "new set vs every existing set" of
// many queries at once).  One warp per listed pair: box test, then the LP from the middle of the overlap.
__global__ void __launch_bounds__(256) k_pair_list(const double* __restrict__ A, const double* __restrict__ b,
                                                   const int* __restrict__ m, int m_max, double tol,
                                                   const double* __restrict__ aabb, const int2* __restrict__ pairs,
                                                   int P, int* __restrict__ result, double* __restrict__ x_feas) {
  __shared__ double scratch[8][BP_LP_SCRATCH_DOUBLES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int p = blockIdx.x * 8 + wib;
  if (p >= P) return;
  const int2 pr = pairs[p];
  bool apart = false, have_region = true;
  double x0[3], region[6];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double loi = __ldg(aabb + (size_t)pr.x * 6 + k), hii = __ldg(aabb + (size_t)pr.x * 6 + 3 + k);
    const double loj = __ldg(aabb + (size_t)pr.y * 6 + k), hij = __ldg(aabb + (size_t)pr.y * 6 + 3 + k);
    if (loi > hij + BP_AABB_EPS || loj > hii + BP_AABB_EPS) apart = true;
    x0[k] = 0.5 * (fmax(loi, loj) + fmin(hii, hij));
    if (!(fabs(x0[k]) < 1e6)) x0[k] = 0.0;
    region[k] = fmax(loi, loj) - BP_AABB_EPS; region[3 + k] = fmin(hii, hij) + BP_AABB_EPS;
    have_region = have_region && fabs(region[k]) < 1e6 && fabs(region[3 + k]) < 1e6;
  }
  int res = 0;
  double xi[3] = {0.0, 0.0, 0.0};
  if (!apart)
    apart = bp_pair_margin_reject(A + (size_t)pr.x * m_max * 3, b + (size_t)pr.x * m_max, m[pr.x],
                                  aabb + (size_t)pr.x * 6, A + (size_t)pr.y * m_max * 3, b + (size_t)pr.y * m_max,
                                  m[pr.y], aabb + (size_t)pr.y * 6, tol);
  if (!apart)
    res = bp_pair_feasible_warp(A + (size_t)pr.x * m_max * 3, b + (size_t)pr.x * m_max, m[pr.x],
                                A + (size_t)pr.y * m_max * 3, b + (size_t)pr.y * m_max, m[pr.y], tol, scratch[wib],
                                nullptr, xi, x0, BP_LP_T0_SCALE, have_region ? region : nullptr);
  if (lane == 0) {
    result[p] = res;
    if (x_feas) { x_feas[3 * (size_t)p] = xi[0]; x_feas[3 * (size_t)p + 1] = xi[1]; x_feas[3 * (size_t)p + 2] = xi[2]; }
  }
}

// ---------------------------------------------------------------------------
// Set-obstacle hit test (bp_sets_obstacles): which obstacle of its scene, if any, does a planned set meet after the
// obstacles moved?  Set s is hit by obstacle o when set_intersection([A_s, b_s], [A_o, b_o], tol) succeeds -- the
// decision of an edge of the set graph.  The obstacle rows are the scene's: box o gives [I; -I] x <= [ub; -lb] from
// the inflated columns (make_box + obs_size_increase, bit for bit: -(lb - r) == -lb + r in fp64), a polytope its
// nrows[o] rows.  One warp per set walks its scene's obstacles in index order, 32 at a time: every lane tests one
// obstacle's box against the set's (k_set_aabb), the survivors go through the warp LP one after another in index
// order, and the warp stops at the first hit, which is then the lowest index.
// ---------------------------------------------------------------------------
// rows of the set, then of obstacle o (box or polytope), every offset shrunk by tol
struct BpSetObstacleRows {
  const double *As, *bs;
  int ms;
  const double* prow;    // [nrows, 4] rows of a polytope obstacle, or NULL: the box lo[3] | hi[3] at box
  const double* box;
  double tol;
  __device__ __forceinline__ void operator()(int i, double* a, double& c) const {
    if (i < ms) {
      a[0] = As[3 * i]; a[1] = As[3 * i + 1]; a[2] = As[3 * i + 2];
      c = bs[i] - tol;
      return;
    }
    const int r = i - ms;
    if (prow) {
      a[0] = prow[4 * r]; a[1] = prow[4 * r + 1]; a[2] = prow[4 * r + 2];
      c = prow[4 * r + 3] - tol;
      return;
    }
    const int k = r < 3 ? r : r - 3;
    const double sg = r < 3 ? 1.0 : -1.0;
    a[0] = k == 0 ? sg : 0.0; a[1] = k == 1 ? sg : 0.0; a[2] = k == 2 ? sg : 0.0;
    c = (r < 3 ? box[3 + k] : -box[k]) - tol;
  }
};

// (the boxes, the start point and the region of the LP live in shared memory: held in registers next to the
// two-rows-per-lane LP they spilled)
__global__ void __launch_bounds__(256) k_sets_obstacles(SceneView sc, int n_scenes, const int* __restrict__ set_scene,
                                                        const double* __restrict__ A, const double* __restrict__ b,
                                                        const int* __restrict__ m, int S, int m_max, double tol,
                                                        const double* __restrict__ aabb, int* __restrict__ first_hit) {
  __shared__ double scratch[8][BP_LP_SCRATCH_DOUBLES];
  __shared__ double boxes[8][24];    // set box [0, 6) | obstacle box [6, 12) | LP region [12, 18) | start point [18, 21)
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int s = blockIdx.x * 8 + wib;
  if (s >= S) return;
  const int k = set_scene ? set_scene[s] : 0;
  if (k < 0 || k >= n_scenes) {
    if (lane == 0) first_hit[s] = -2;
    return;
  }
  const int o0 = sc.seg_off ? sc.seg_off[k] : 0;
  const int n = sc.seg_off ? sc.seg_off[k + 1] - o0 : sc.n;
  double* wb = boxes[wib];
  if (lane < 6) wb[lane] = __ldg(aabb + (size_t)s * 6 + lane);
  // this lane's axis (lanes 0-2) of the obstacle columns
  const int ax = lane < 3 ? lane : 0;
  const double* lb = ax == 0 ? sc.lb[0] : (ax == 1 ? sc.lb[1] : sc.lb[2]);
  const double* ub = ax == 0 ? sc.ub[0] : (ax == 1 ? sc.ub[1] : sc.ub[2]);
  __syncwarp();
  BpSetObstacleRows rows;
  rows.As = A + (size_t)s * m_max * 3;
  rows.bs = b + (size_t)s * m_max;
  rows.ms = min(max(m[s], 0), m_max);
  rows.box = wb + 6;
  rows.tol = tol;
  int hit = -1;
  for (int base = 0; base < n && hit < 0; base += 32) {
    const int j = base + lane;
    bool keep = false;
    if (j < n) {
      keep = true;
#pragma unroll
      for (int e = 0; e < 3; ++e) {
        const double lo = __ldg(sc.lb[e] + o0 + j), hi = __ldg(sc.ub[e] + o0 + j);
        if (wb[e] > hi + BP_AABB_EPS || lo > wb[3 + e] + BP_AABB_EPS) keep = false;
      }
    }
    unsigned int mask = __ballot_sync(full, keep);
    while (mask && hit < 0) {
      const int f = __ffs(mask) - 1;
      mask &= mask - 1u;
      const int o = o0 + base + f;
      bool finite = true;
      if (lane < 3) {
        const double olo = __ldg(lb + o), ohi = __ldg(ub + o);
        const double lo = fmax(wb[lane], olo), hi = fmin(wb[3 + lane], ohi);
        const double x0 = 0.5 * (lo + hi);
        wb[6 + lane] = olo; wb[9 + lane] = ohi;
        wb[12 + lane] = lo - BP_AABB_EPS; wb[15 + lane] = hi + BP_AABB_EPS;   // every common point lies in this box
        wb[18 + lane] = fabs(x0) < 1e6 ? x0 : 0.0;                          // start at the middle of the overlap
        finite = fabs(lo) < 1e6 && fabs(hi) < 1e6;
      }
      const bool have_region = __all_sync(full, finite);
      __syncwarp();
      rows.prow = sc.rows ? sc.rows + (size_t)o * BP_OBS_ROWS * 4 : nullptr;
      const int mt = rows.ms + (sc.rows ? __ldg(sc.nrows + o) : 6);
      const double* reg = have_region ? wb + 12 : nullptr;
      // at most 48 + 15 rows: one or two rows per lane
      const int res = mt <= 32 ? bp_lp_feasible_warp_impl<1>(rows, mt, scratch[wib], nullptr, nullptr, wb + 18,
                                                              BP_LP_T0_SCALE, reg)
                               : bp_lp_feasible_warp_impl<2>(rows, mt, scratch[wib], nullptr, nullptr, wb + 18,
                                                              BP_LP_T0_SCALE, reg);
      if (res) hit = base + f;
      __syncwarp();
    }
  }
  if (lane == 0) first_hit[s] = hit;
}

// ---------------------------------------------------------------------------
// K8 ("next" row 1): redundancy removal of a set's rows.
// Replaces reduce_ineqs (bound_planner/utils/util_functions.py:82-88; cddlib
// dd_MatrixRedundancyRemove): a row is kept iff it supports a facet, i.e. the
// polytope has three non-collinear vertices on it.  One 128-thread CTA per set:
// phase 1 enumerates the vertices (all row triples, as k_set_aabb) into shared
// memory; phase 2, one thread per row, measures the spread of the vertices on
// its plane; of two identical planes the later row goes (cddlib walks the rows
// from the last to the first and removes on the spot).  Kept rows keep their
// order and coefficients.
// ---------------------------------------------------------------------------
#define BP_RED_VMAX 768
#define BP_RED_ON_FACE 1e-8
#define BP_RED_SPREAD 1e-7

__global__ void __launch_bounds__(128) k_reduce_rows(const double* __restrict__ A, const double* __restrict__ b,
                                                     const int* __restrict__ m, int m_max, double* __restrict__ A_out,
                                                     double* __restrict__ b_out, int* __restrict__ m_out,
                                                     unsigned char* __restrict__ keep_out, int* __restrict__ status) {
  __shared__ double sA[BP_MAX_ROWS * 3], sb[BP_MAX_ROWS];
  __shared__ double sv[BP_RED_VMAX * 3];
  __shared__ int nverts;
  __shared__ unsigned char skeep[BP_MAX_ROWS];
  const int s = blockIdx.x, tid = threadIdx.x;
  const int ms = m[s];
  for (int e = tid; e < ms * 3; e += 128) sA[e] = A[(size_t)s * m_max * 3 + e];
  for (int e = tid; e < ms; e += 128) sb[e] = b[(size_t)s * m_max + e];
  if (tid == 0) nverts = 0;
  __syncthreads();
  const int ntrip = ms * (ms - 1) * (ms - 2) / 6;
  for (int t = tid; t < ntrip; t += 128) {
    int i = 0, rem = t;
    for (;;) { const int c = (ms - 1 - i) * (ms - 2 - i) / 2; if (rem < c) break; rem -= c; ++i; }
    int j = i + 1;
    for (;;) { const int c = ms - 1 - j; if (rem < c) break; rem -= c; ++j; }
    const int k = j + 1 + rem;
    const double a0 = sA[3 * i], a1 = sA[3 * i + 1], a2 = sA[3 * i + 2], ab = sb[i];
    const double c0 = sA[3 * j], c1 = sA[3 * j + 1], c2 = sA[3 * j + 2], cb = sb[j];
    const double d0 = sA[3 * k], d1 = sA[3 * k + 1], d2 = sA[3 * k + 2], db = sb[k];
    const double n0 = a1 * c2 - a2 * c1, n1 = a2 * c0 - a0 * c2, n2 = a0 * c1 - a1 * c0;
    const double det = n0 * d0 + n1 * d1 + n2 * d2;
    const double scale = (fabs(n0) + fabs(n1) + fabs(n2)) * (fabs(d0) + fabs(d1) + fabs(d2));
    if (!(fabs(det) > 1e-12 * scale)) continue;
    const double e0 = c1 * d2 - c2 * d1, e1 = c2 * d0 - c0 * d2, e2 = c0 * d1 - c1 * d0;
    const double f0 = d1 * a2 - d2 * a1, f1 = d2 * a0 - d0 * a2, f2 = d0 * a1 - d1 * a0;
    const double id = 1.0 / det;
    const double v0 = (ab * e0 + cb * f0 + db * n0) * id;
    const double v1 = (ab * e1 + cb * f1 + db * n1) * id;
    const double v2 = (ab * e2 + cb * f2 + db * n2) * id;
    bool inside = true;
    for (int r = 0; r < ms; ++r) {
      const double q0 = sA[3 * r], q1 = sA[3 * r + 1], q2 = sA[3 * r + 2];
      const double viol = q0 * v0 + q1 * v1 + q2 * v2 - sb[r];
      if (viol > BP_AABB_EPS * (1.0 + fabs(q0 * v0) + fabs(q1 * v1) + fabs(q2 * v2))) inside = false;
    }
    if (inside) {
      const int slot = atomicAdd(&nverts, 1);
      if (slot < BP_RED_VMAX) { sv[3 * slot] = v0; sv[3 * slot + 1] = v1; sv[3 * slot + 2] = v2; }
    }
  }
  __syncthreads();
  const int nv = nverts < BP_RED_VMAX ? nverts : BP_RED_VMAX;
  const bool overflow = nverts > BP_RED_VMAX;
  if (tid < ms) {
    const int r = tid;
    const double q0 = sA[3 * r], q1 = sA[3 * r + 1], q2 = sA[3 * r + 2], qb = sb[r];
    const double qn = sqrt(q0 * q0 + q1 * q1 + q2 * q2);
    bool keep = true;
    if (!(qn > 0.0)) keep = qb < 0.0;                 // 0 <= b is always implied
    else if (!overflow) {
      // the later of two identical planes is redundant
      for (int e = 0; e < r && keep; ++e) {
        const double en = sqrt(sA[3 * e] * sA[3 * e] + sA[3 * e + 1] * sA[3 * e + 1] + sA[3 * e + 2] * sA[3 * e + 2]);
        if (en > 0.0 && fabs(sA[3 * e] / en - q0 / qn) <= 1e-12 && fabs(sA[3 * e + 1] / en - q1 / qn) <= 1e-12 &&
            fabs(sA[3 * e + 2] / en - q2 / qn) <= 1e-12 && fabs(sb[e] / en - qb / qn) <= 1e-12)
          keep = false;
      }
      if (keep) {
        // spread of the vertices lying on the plane of row r: point, segment or polygon?
        const double tolf = BP_RED_ON_FACE * (qn + fabs(qb));
        int first = -1;
        for (int v = 0; v < nv && first < 0; ++v)
          if (fabs(q0 * sv[3 * v] + q1 * sv[3 * v + 1] + q2 * sv[3 * v + 2] - qb) <= tolf) first = v;
        if (first < 0) keep = false;
        else {
          const double p0 = sv[3 * first], p1 = sv[3 * first + 1], p2 = sv[3 * first + 2];
          double dmax = 0.0, w0 = 0.0, w1 = 0.0, w2 = 0.0;
          for (int v = 0; v < nv; ++v) {
            const double x0 = sv[3 * v], x1 = sv[3 * v + 1], x2 = sv[3 * v + 2];
            if (fabs(q0 * x0 + q1 * x1 + q2 * x2 - qb) > tolf) continue;
            const double dd = (x0 - p0) * (x0 - p0) + (x1 - p1) * (x1 - p1) + (x2 - p2) * (x2 - p2);
            if (dd > dmax) { dmax = dd; w0 = x0 - p0; w1 = x1 - p1; w2 = x2 - p2; }
          }
          if (!(dmax > BP_RED_SPREAD * BP_RED_SPREAD)) keep = false;      // the plane touches in a point
          else {
            double amax = 0.0;
            for (int v = 0; v < nv; ++v) {
              const double x0 = sv[3 * v], x1 = sv[3 * v + 1], x2 = sv[3 * v + 2];
              if (fabs(q0 * x0 + q1 * x1 + q2 * x2 - qb) > tolf) continue;
              const double u0 = x0 - p0, u1 = x1 - p1, u2 = x2 - p2;
              const double cx = w1 * u2 - w2 * u1, cy = w2 * u0 - w0 * u2, cz = w0 * u1 - w1 * u0;
              const double ar = cx * cx + cy * cy + cz * cz;
              amax = ar > amax ? ar : amax;
            }
            if (!(amax > BP_RED_SPREAD * BP_RED_SPREAD * dmax)) keep = false;   // ... or along an edge
          }
        }
      }
    }
    skeep[r] = keep ? 1 : 0;
  }
  __syncthreads();
  if (tid == 0) {
    int k = 0;
    double* Ao = A_out + (size_t)s * m_max * 3;
    double* bo = b_out + (size_t)s * m_max;
    for (int r = 0; r < ms; ++r) {
      if (keep_out) keep_out[(size_t)s * m_max + r] = skeep[r];
      if (skeep[r]) {
        Ao[3 * k] = sA[3 * r]; Ao[3 * k + 1] = sA[3 * r + 1]; Ao[3 * k + 2] = sA[3 * r + 2];
        bo[k] = sb[r];
        ++k;
      }
    }
    for (int r = k; r < m_max; ++r) { Ao[3 * r] = 0.0; Ao[3 * r + 1] = 0.0; Ao[3 * r + 2] = 0.0; bo[r] = 10.0; }
    if (keep_out) for (int r = ms; r < m_max; ++r) keep_out[(size_t)s * m_max + r] = 0;
    m_out[s] = k;
    if (status) status[s] = overflow ? BP_ROW_OVERFLOW : BP_OK;
  }
}

// ---------------------------------------------------------------------------
// Vertex enumeration of polytopes {A x <= b} (SURVEY 8f row 4): replaces compute_polytope_vertices
// (bound_planner/utils/util_functions.py:66-79; cddlib double description) -- what add_obstacle_reps needs to
// turn obstacle halfspace sets into the vertex lists of obs_points_sets (BoundPlanner.py:142).  One 128-thread
// CTA per set: every row triple gives a candidate point (as in k_set_aabb / k_reduce_rows); the feasible ones are
// kept, coinciding candidates (more than three planes through a vertex) merged, and the vertices written in the
// order of their first triple (deterministic).  status: BP_OK, BP_NOT_A_POLYTOPE (the recession cone
// {d : A d <= 0} is not {0}: the reference raises ValueError("Polyhedron is not a polytope")), BP_ROW_OVERFLOW
// (more than vmax vertices).
// ---------------------------------------------------------------------------
#define BP_VERT_MERGE 1e-9
// The vertices of one polytope {x : sA x <= sb} (ms rows in shared memory) by one 128-thread CTA: V[vmax,3] of the
// set, *nv_out and the returned status are written by thread 0 (the return value is valid there only).
__device__ __forceinline__ int polytope_vertices_cta(const double* sA, const double* sb, int ms, int vmax,
                                                     double* __restrict__ V, int* __restrict__ nv_out) {
  __shared__ double sv[BP_RED_VMAX * 3];
  __shared__ int st[BP_RED_VMAX];                   // triple index of every stored candidate
  __shared__ unsigned char dup[BP_RED_VMAX];
  __shared__ int nverts, unbounded, anypair;
  const int tid = threadIdx.x;
  if (tid == 0) { nverts = 0; unbounded = 0; anypair = 0; }
  __syncthreads();
  // bounded?  a direction of the recession cone, if there is one, can be taken along +-(a_i x a_j)
  for (int t = tid; t < ms * ms; t += 128) {
    const int i = t / ms, j = t % ms;
    if (j <= i) continue;
    double d0 = sA[3 * i + 1] * sA[3 * j + 2] - sA[3 * i + 2] * sA[3 * j + 1];
    double d1 = sA[3 * i + 2] * sA[3 * j] - sA[3 * i] * sA[3 * j + 2];
    double d2 = sA[3 * i] * sA[3 * j + 1] - sA[3 * i + 1] * sA[3 * j];
    const double dn = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
    const double ni = sqrt(sA[3 * i] * sA[3 * i] + sA[3 * i + 1] * sA[3 * i + 1] + sA[3 * i + 2] * sA[3 * i + 2]);
    const double nj = sqrt(sA[3 * j] * sA[3 * j] + sA[3 * j + 1] * sA[3 * j + 1] + sA[3 * j + 2] * sA[3 * j + 2]);
    if (!(dn > 1e-12 * ni * nj)) continue;          // parallel (or zero) rows
    anypair = 1;
    d0 /= dn; d1 /= dn; d2 /= dn;
    double mx = -BP_INF, mn = BP_INF;
    for (int r = 0; r < ms; ++r) {
      const double rn = sqrt(sA[3 * r] * sA[3 * r] + sA[3 * r + 1] * sA[3 * r + 1] + sA[3 * r + 2] * sA[3 * r + 2]);
      if (!(rn > 0.0)) continue;
      const double v = (sA[3 * r] * d0 + sA[3 * r + 1] * d1 + sA[3 * r + 2] * d2) / rn;
      mx = fmax(mx, v); mn = fmin(mn, v);
    }
    if (mx <= 1e-12 || mn >= -1e-12) unbounded = 1;   // A d <= 0 for d or for -d
  }
  const int ntrip = ms * (ms - 1) * (ms - 2) / 6;
  for (int t = tid; t < ntrip; t += 128) {
    int i = 0, rem = t;
    for (;;) { const int c = (ms - 1 - i) * (ms - 2 - i) / 2; if (rem < c) break; rem -= c; ++i; }
    int j = i + 1;
    for (;;) { const int c = ms - 1 - j; if (rem < c) break; rem -= c; ++j; }
    const int k = j + 1 + rem;
    const double a0 = sA[3 * i], a1 = sA[3 * i + 1], a2 = sA[3 * i + 2], ab = sb[i];
    const double c0 = sA[3 * j], c1 = sA[3 * j + 1], c2 = sA[3 * j + 2], cb = sb[j];
    const double d0 = sA[3 * k], d1 = sA[3 * k + 1], d2 = sA[3 * k + 2], db = sb[k];
    const double n0 = a1 * c2 - a2 * c1, n1 = a2 * c0 - a0 * c2, n2 = a0 * c1 - a1 * c0;
    const double det = n0 * d0 + n1 * d1 + n2 * d2;
    const double scale = (fabs(n0) + fabs(n1) + fabs(n2)) * (fabs(d0) + fabs(d1) + fabs(d2));
    if (!(fabs(det) > 1e-12 * scale)) continue;
    const double e0 = c1 * d2 - c2 * d1, e1 = c2 * d0 - c0 * d2, e2 = c0 * d1 - c1 * d0;
    const double f0 = d1 * a2 - d2 * a1, f1 = d2 * a0 - d0 * a2, f2 = d0 * a1 - d1 * a0;
    const double id = 1.0 / det;
    const double v0 = (ab * e0 + cb * f0 + db * n0) * id;
    const double v1 = (ab * e1 + cb * f1 + db * n1) * id;
    const double v2 = (ab * e2 + cb * f2 + db * n2) * id;
    bool inside = true;
    for (int r = 0; r < ms; ++r) {
      const double q0 = sA[3 * r], q1 = sA[3 * r + 1], q2 = sA[3 * r + 2];
      const double viol = q0 * v0 + q1 * v1 + q2 * v2 - sb[r];
      if (viol > BP_AABB_EPS * (1.0 + fabs(q0 * v0) + fabs(q1 * v1) + fabs(q2 * v2))) inside = false;
    }
    if (inside) {
      const int slot = atomicAdd(&nverts, 1);
      if (slot < BP_RED_VMAX) { sv[3 * slot] = v0; sv[3 * slot + 1] = v1; sv[3 * slot + 2] = v2; st[slot] = t; }
    }
  }
  __syncthreads();
  const int nc = nverts < BP_RED_VMAX ? nverts : BP_RED_VMAX;
  // a candidate is a duplicate when a candidate of a smaller triple index lies at the same point
  for (int v = tid; v < nc; v += 128) {
    bool d = false;
    const double scl = 1.0 + fabs(sv[3 * v]) + fabs(sv[3 * v + 1]) + fabs(sv[3 * v + 2]);
    for (int u = 0; u < nc && !d; ++u)
      if (st[u] < st[v] && fabs(sv[3 * u] - sv[3 * v]) + fabs(sv[3 * u + 1] - sv[3 * v + 1]) +
                               fabs(sv[3 * u + 2] - sv[3 * v + 2]) <= BP_VERT_MERGE * scl)
        d = true;
    dup[v] = d ? 1 : 0;
  }
  __syncthreads();
  __shared__ int n_unique;
  if (tid == 0) n_unique = 0;
  __syncthreads();
  for (int v = tid; v < nc; v += 128) {
    if (dup[v]) continue;
    int rank = 0;
    for (int u = 0; u < nc; ++u) rank += (!dup[u] && st[u] < st[v]) ? 1 : 0;
    atomicAdd(&n_unique, 1);
    if (rank < vmax) {
      double* o = V + (size_t)rank * 3;
      o[0] = sv[3 * v]; o[1] = sv[3 * v + 1]; o[2] = sv[3 * v + 2];
    }
  }
  __syncthreads();
  int stt = BP_OK;
  if (tid == 0) {
    const int nu = n_unique;
    *nv_out = nu < vmax ? nu : vmax;
    if (unbounded || !anypair || nu == 0) stt = BP_NOT_A_POLYTOPE;
    else if (nverts > BP_RED_VMAX || nu > vmax) stt = BP_ROW_OVERFLOW;
  }
  return stt;
}

__global__ void __launch_bounds__(128) k_polytope_vertices(const double* __restrict__ A, const double* __restrict__ b,
                                                           const int* __restrict__ m, int m_max, int vmax,
                                                           double* __restrict__ V, int* __restrict__ nv_out,
                                                           int* __restrict__ status) {
  __shared__ double sA[BP_MAX_ROWS * 3], sb[BP_MAX_ROWS];
  const int s = blockIdx.x, tid = threadIdx.x;
  const int ms = m[s];
  for (int e = tid; e < ms * 3; e += 128) sA[e] = A[(size_t)s * m_max * 3 + e];
  for (int e = tid; e < ms; e += 128) sb[e] = b[(size_t)s * m_max + e];
  const int stt = polytope_vertices_cta(sA, sb, ms, vmax, V + (size_t)s * vmax * 3, nv_out + s);
  if (tid == 0) status[s] = stt;
}

// ---------------------------------------------------------------------------
// K9 ("next" row 2, part 1): does the end effector fit into an intersection set?
// Replaces BoundPlanner.check_intersection (BoundPlanner.py:745-772): for omega_k =
// k/19, k = 0..19, l_k = Rodrigues(omega_hat, |omega| omega_k) l_ee (rotated on the
// host, optimization_functions.py:83-104); the qpOASES feasibility QP (J = 0,
// optimization_functions.py:140-183) of  A p <= b - 0.001,  A (p + l_k) <= b - 0.001
// is the same phase-I LP as K6 on the doubled row set.  First feasible k wins.
// One warp per (set i, set j) pair of the work list; rows = rows of i then rows of j.
// ---------------------------------------------------------------------------
#define BP_FIT_SAMPLES 20
struct FitParams {
  double l[BP_FIT_SAMPLES][3];    // rotated end-effector offsets
  double margin;                  // 0.001 (:746)
  int n_samples;
  int nu;                         // number of distinct offsets
  int uidx[BP_FIT_SAMPLES];       // first sample index of every distinct offset, ascending
};

struct BpFitRows {
  const double *A1, *b1, *A2, *b2;
  int m1, mtot;                   // mtot = m1 + m2; rows [mtot, 2 mtot) are the shifted copies
  double l0, l1, l2, margin;
  __device__ __forceinline__ void operator()(int i, double* a, double& c) const {
    const int r = i < mtot ? i : i - mtot;
    const double* A = r < m1 ? A1 + 3 * r : A2 + 3 * (r - m1);
    a[0] = A[0]; a[1] = A[1]; a[2] = A[2];
    c = (r < m1 ? b1[r] : b2[r - m1]) - margin;
    if (i >= mtot) c -= a[0] * l0 + a[1] * l1 + a[2] * l2;      // A (p + l) <= b - margin
  }
};

// One warp per (pair, DISTINCT end-effector offset): the reference walks its 20 rotations one after the other and
// stops at the first that fits (:745-772); here they are tested side by side and the smallest fitting index wins
// (atomicMin), so a pair that does not fit costs one LP latency instead of twenty.  Offsets that repeat (no
// rotation between start and end: all 20 are the same vector) are tested once: fp.uidx lists the first index of
// every distinct offset.  first_sample must be preset to 0x7f7f7f7f; k_fit_finish turns it into the outputs.
__global__ void __launch_bounds__(256) k_fit_check(const double* __restrict__ A, const double* __restrict__ b,
                                                   const int* __restrict__ m, int m_max, const int2* __restrict__ pairs,
                                                   int P, const double* __restrict__ x0s,
                                                   const int* __restrict__ active, FitParams fp,
                                                   int* __restrict__ first_sample) {
  __shared__ double scratch[8][BP_LP_SCRATCH_DOUBLES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int w = blockIdx.x * 8 + wib;
  const int p = w / fp.nu;
  if (p >= P) return;
  if (active && !active[p]) return;            // e.g. the pair does not intersect: no fit check
  const int k = fp.uidx[w - p * fp.nu];
  const int2 pr = pairs[p];
  const int m1 = m[pr.x], m2 = (pr.y == pr.x) ? 0 : m[pr.y];     // i == j: a single set
  const int mtot = m1 + m2;
  if (2 * mtot > 96) return;                   // (bp_lp_feasible_warp takes at most 96 rows; k_fit_finish flags it)
  double x0[3] = {0.0, 0.0, 0.0};
  if (x0s) { x0[0] = x0s[3 * p]; x0[1] = x0s[3 * p + 1]; x0[2] = x0s[3 * p + 2]; }
  BpFitRows rows{A + (size_t)pr.x * m_max * 3, b + (size_t)pr.x * m_max, A + (size_t)pr.y * m_max * 3,
                 b + (size_t)pr.y * m_max, m1, mtot, fp.l[k][0], fp.l[k][1], fp.l[k][2], fp.margin};
  const int ok = bp_lp_feasible_warp(rows, 2 * mtot, scratch[wib], nullptr, nullptr, x0, BP_LP_T0_SCALE);
  if (ok && lane == 0) atomicMin(first_sample + p, k);
}

__global__ void k_fit_finish(const int* __restrict__ m, const int2* __restrict__ pairs, int P,
                             const int* __restrict__ active, int n_samples, int* __restrict__ fits,
                             int* __restrict__ first_sample) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  int found = first_sample[p];
  if (found < 0 || found >= n_samples) found = -1;
  if (active && !active[p]) found = -1;
  else {
    const int2 pr = pairs[p];
    const int mtot = m[pr.x] + ((pr.y == pr.x) ? 0 : m[pr.y]);
    if (2 * mtot > 96) found = -2;                              // too many rows for one warp
  }
  fits[p] = found >= 0 ? 1 : (found == -2 ? -1 : 0);
  first_sample[p] = found;
}

// ---------------------------------------------------------------------------
// K10 ("next" row 2, part 2): projection of a point onto an intersection set.
// Replaces the qpOASES projection QP of add_edges (BoundPlanner.py:842-864; problem
// optimization_functions.py:107-137):  min |x - x_d|^2  s.t.  [A_i; A_j] x <= [b_i; b_j].
// Exact: the projection is the projection onto the affine hull of its <= 3 active rows;
// one warp per pair enumerates all active sets of size 0..3 (lanes stride the
// candidates), keeps the feasible ones and takes the closest.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_project(const double* __restrict__ A, const double* __restrict__ b,
                                                 const int* __restrict__ m, int m_max, const int2* __restrict__ pairs,
                                                 int P, const double* __restrict__ xd, double* __restrict__ xout,
                                                 int* __restrict__ status, const int* __restrict__ act_a = nullptr,
                                                 const int* __restrict__ act_b = nullptr) {
  __shared__ double sA[8][2 * BP_MAX_ROWS * 3], sb[8][2 * BP_MAX_ROWS];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int p = blockIdx.x * 8 + wib;
  if (p >= P) return;
  if ((act_a && !act_a[p]) || (act_b && !act_b[p])) {       // gated off (e.g. the pair does not intersect)
    if (lane == 0 && status) status[p] = -1;
    return;
  }
  const int2 pr = pairs[p];
  const int m1 = m[pr.x], m2 = (pr.y == pr.x) ? 0 : m[pr.y];
  const int mt = m1 + m2;
  double* rA = sA[wib];
  double* rb = sb[wib];
  const double d0 = xd[3 * p], d1 = xd[3 * p + 1], d2 = xd[3 * p + 2];
  for (int r = lane; r < mt; r += 32) {
    const double* Ar = r < m1 ? A + ((size_t)pr.x * m_max + r) * 3 : A + ((size_t)pr.y * m_max + (r - m1)) * 3;
    const double br = r < m1 ? b[(size_t)pr.x * m_max + r] : b[(size_t)pr.y * m_max + (r - m1)];
    rA[3 * r] = Ar[0]; rA[3 * r + 1] = Ar[1]; rA[3 * r + 2] = Ar[2];
    rb[r] = br - (Ar[0] * d0 + Ar[1] * d1 + Ar[2] * d2);         // shift: z = x - x_d, rows A z <= b - A x_d
  }
  __syncwarp();
  double best = BP_INF, z0 = 0.0, z1 = 0.0, z2 = 0.0;
  auto feasible = [&](double a, double c, double e) {
    bool ok = true;
    for (int r = 0; r < mt; ++r) {
      const double q0 = rA[3 * r], q1 = rA[3 * r + 1], q2 = rA[3 * r + 2];
      const double v = q0 * a + q1 * c + q2 * e - rb[r];
      if (v > 1e-10 * (1.0 + fabs(rb[r]) + fabs(q0 * a) + fabs(q1 * c) + fabs(q2 * e))) ok = false;
    }
    return ok;
  };
  auto consider = [&](double a, double c, double e) {
    const double n2 = a * a + c * c + e * e;
    if (n2 < best && feasible(a, c, e)) { best = n2; z0 = a; z1 = c; z2 = e; }
  };
  if (lane == 0) consider(0.0, 0.0, 0.0);                        // x_d already inside
  // one active row: z = a h / |a|^2
  for (int i = lane; i < mt; i += 32) {
    const double a0 = rA[3 * i], a1 = rA[3 * i + 1], a2 = rA[3 * i + 2];
    const double nn = a0 * a0 + a1 * a1 + a2 * a2;
    if (nn > 0.0) { const double t = rb[i] / nn; consider(a0 * t, a1 * t, a2 * t); }
  }
  // two active rows: z = lam_i a_i + lam_j a_j with the 2x2 Gram system
  const int np2 = mt * (mt - 1) / 2;
  for (int t = lane; t < np2; t += 32) {
    int i = 0, rem = t;
    while (rem >= mt - 1 - i) { rem -= mt - 1 - i; ++i; }
    const int j = i + 1 + rem;
    const double a0 = rA[3 * i], a1 = rA[3 * i + 1], a2 = rA[3 * i + 2];
    const double c0 = rA[3 * j], c1 = rA[3 * j + 1], c2 = rA[3 * j + 2];
    const double gaa = a0 * a0 + a1 * a1 + a2 * a2, gcc = c0 * c0 + c1 * c1 + c2 * c2;
    const double gac = a0 * c0 + a1 * c1 + a2 * c2;
    const double det = gaa * gcc - gac * gac;
    if (!(det > 1e-12 * gaa * gcc)) continue;
    const double li = (rb[i] * gcc - rb[j] * gac) / det, lj = (rb[j] * gaa - rb[i] * gac) / det;
    consider(li * a0 + lj * c0, li * a1 + lj * c1, li * a2 + lj * c2);
  }
  // three active rows: the vertex of the three planes
  const int np3 = mt * (mt - 1) * (mt - 2) / 6;
  for (int t = lane; t < np3; t += 32) {
    int i = 0, rem = t;
    for (;;) { const int c = (mt - 1 - i) * (mt - 2 - i) / 2; if (rem < c) break; rem -= c; ++i; }
    int j = i + 1;
    for (;;) { const int c = mt - 1 - j; if (rem < c) break; rem -= c; ++j; }
    const int k = j + 1 + rem;
    const double a0 = rA[3 * i], a1 = rA[3 * i + 1], a2 = rA[3 * i + 2], ab = rb[i];
    const double c0 = rA[3 * j], c1 = rA[3 * j + 1], c2 = rA[3 * j + 2], cb = rb[j];
    const double e0 = rA[3 * k], e1 = rA[3 * k + 1], e2 = rA[3 * k + 2], eb = rb[k];
    const double n0 = a1 * c2 - a2 * c1, n1 = a2 * c0 - a0 * c2, n2 = a0 * c1 - a1 * c0;
    const double det = n0 * e0 + n1 * e1 + n2 * e2;
    const double scale = (fabs(n0) + fabs(n1) + fabs(n2)) * (fabs(e0) + fabs(e1) + fabs(e2));
    if (!(fabs(det) > 1e-12 * scale)) continue;
    const double f0 = c1 * e2 - c2 * e1, f1 = c2 * e0 - c0 * e2, f2 = c0 * e1 - c1 * e0;
    const double g0 = e1 * a2 - e2 * a1, g1 = e2 * a0 - e0 * a2, g2 = e0 * a1 - e1 * a0;
    const double id = 1.0 / det;
    consider((ab * f0 + cb * g0 + eb * n0) * id, (ab * f1 + cb * g1 + eb * n1) * id, (ab * f2 + cb * g2 + eb * n2) * id);
  }
  // warp argmin (ties -> lowest lane: the point is unique)
  double bv = best;
  int bl = lane;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, off);
    const int ol = __shfl_xor_sync(0xffffffffu, bl, off);
    if (ov < bv || (ov == bv && ol < bl)) { bv = ov; bl = ol; }
  }
  z0 = __shfl_sync(0xffffffffu, z0, bl); z1 = __shfl_sync(0xffffffffu, z1, bl); z2 = __shfl_sync(0xffffffffu, z2, bl);
  if (lane == 0) {
    xout[3 * p] = d0 + z0; xout[3 * p + 1] = d1 + z1; xout[3 * p + 2] = d2 + z2;
    if (status) status[p] = bv < BP_INF ? BP_OK : BP_MVIE_NO_INTERIOR;      // empty intersection
  }
}

// ---------------------------------------------------------------------------
// K7: FK, one thread per configuration, 128 configurations per CTA.
// HBM-bound streaming kernel: the q tile comes in and the result tiles go out
// through shared memory with TMA bulk copies (cp.async.bulk, one elected
// thread, mbarrier completion) so that every global transaction is a full
// line and no LSU instructions are spent on staging; a plain coalesced loop
// handles a ragged last tile or unaligned pointers.
// ---------------------------------------------------------------------------
#define FK_T 128

template <bool POSE, bool JAC>
__global__ void __launch_bounds__(FK_T) k_fk(const double* __restrict__ q, int B, double* __restrict__ p_ee,
                                             double* __restrict__ p_col, double* __restrict__ T_ee,
                                             double* __restrict__ jac, int use_tma) {
  extern __shared__ __align__(128) double s_fk[];
  __shared__ __align__(8) uint64_t bar;
  double* s_q = s_fk;                       // [FK_T*7]
  double* s_pe = s_q + FK_T * 7;            // [FK_T*3]
  double* s_pc = s_pe + FK_T * 3;           // [FK_T*21]
  double* s_T = s_pc + FK_T * 21;           // [FK_T*16]  (POSE)
  double* s_J = s_T + (POSE ? FK_T * 16 : 0);   // [FK_T*42]  (JAC)
  const int base = blockIdx.x * FK_T;
  const int nb = min(FK_T, B - base);
  const bool bulk = use_tma && nb == FK_T;
  if (bulk) {
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) tma_load_1d(s_q, q + (size_t)base * 7, FK_T * 7 * 8, &bar);
    mbar_wait(&bar, 0);
  } else {
    for (int e = threadIdx.x; e < nb * 7; e += FK_T) s_q[e] = q[(size_t)base * 7 + e];
    __syncthreads();
  }
  if (threadIdx.x < nb) {
    double qq[7], pe[3], pc[21], T[16], J[42];
#pragma unroll
    for (int k = 0; k < 7; ++k) qq[k] = s_q[threadIdx.x * 7 + k];
    bp_fk_iiwa14(qq, pe, pc, POSE ? T : nullptr, JAC ? J : nullptr);
#pragma unroll
    for (int k = 0; k < 3; ++k) s_pe[threadIdx.x * 3 + k] = pe[k];
#pragma unroll
    for (int k = 0; k < 21; ++k) s_pc[threadIdx.x * 21 + k] = pc[k];
    if (POSE) {
#pragma unroll
      for (int k = 0; k < 16; ++k) s_T[threadIdx.x * 16 + k] = T[k];
    }
    if (JAC) {
#pragma unroll
      for (int k = 0; k < 42; ++k) s_J[threadIdx.x * 42 + k] = J[k];
    }
  }
  if (bulk) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy smem writes -> async proxy
    __syncthreads();
    if (threadIdx.x == 0) {
      tma_store_1d(p_ee + (size_t)base * 3, s_pe, FK_T * 3 * 8);
      tma_store_1d(p_col + (size_t)base * 21, s_pc, FK_T * 21 * 8);
      if (POSE) tma_store_1d(T_ee + (size_t)base * 16, s_T, FK_T * 16 * 8);
      if (JAC) tma_store_1d(jac + (size_t)base * 42, s_J, FK_T * 42 * 8);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem must stay valid until read
    }
  } else {
    __syncthreads();
    for (int e = threadIdx.x; e < nb * 3; e += FK_T) p_ee[(size_t)base * 3 + e] = s_pe[e];
    for (int e = threadIdx.x; e < nb * 21; e += FK_T) p_col[(size_t)base * 21 + e] = s_pc[e];
    if (POSE) for (int e = threadIdx.x; e < nb * 16; e += FK_T) T_ee[(size_t)base * 16 + e] = s_T[e];
    if (JAC) for (int e = threadIdx.x; e < nb * 42; e += FK_T) jac[(size_t)base * 42 + e] = s_J[e];
  }
}

// K7b: RobotModel.forward_kinematics (RobotModel.py:70-77): pose, Jacobian and its time derivative for
// (q, dq) pairs, one thread per configuration.  The MPC loop calls this once or twice per step on single
// configurations (MPCNode.py:118, util_functions.py:57), so the outputs (16 + 42 + 42 doubles) are staged through
// shared memory only for coalesced stores; no bulk copies.
__global__ void __launch_bounds__(32) k_fk_kin(const double* __restrict__ q, const double* __restrict__ dq, int B,
                                               double* __restrict__ T_ee, double* __restrict__ jac,
                                               double* __restrict__ djac) {
  __shared__ double s_out[32 * 101];             // odd row stride: conflict-free per-thread rows
  const int base = blockIdx.x * 32;
  const int nb = min(32, B - base);
  if ((int)threadIdx.x < nb) {
    double qq[7], dd[7], pe[3], pc[21], T[16], J[42], dJ[42];
    const size_t i = (size_t)(base + threadIdx.x);
#pragma unroll
    for (int k = 0; k < 7; ++k) { qq[k] = q[i * 7 + k]; dd[k] = dq ? dq[i * 7 + k] : 0.0; }
    bp_fk_iiwa14(qq, pe, pc, T, J, dd, dJ);
    double* o = s_out + threadIdx.x * 101;
#pragma unroll
    for (int k = 0; k < 16; ++k) o[k] = T[k];
#pragma unroll
    for (int k = 0; k < 42; ++k) { o[16 + k] = J[k]; o[58 + k] = dJ[k]; }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < nb * 16; e += 32) T_ee[(size_t)base * 16 + e] = s_out[(e / 16) * 101 + e % 16];
  for (int e = threadIdx.x; e < nb * 42; e += 32) {
    jac[(size_t)base * 42 + e] = s_out[(e / 42) * 101 + 16 + e % 42];
    if (djac) djac[(size_t)base * 42 + e] = s_out[(e / 42) * 101 + 58 + e % 42];
  }
}

// ---------------------------------------------------------------------------
// K11-K13 (SURVEY 8f rows 3-4): the planner loop's own tests, batched over queries.
//   k_sample_filter   the rejection loop of plan_convex_set_path (BoundPlanner.py:459-478): candidate points of a
//                     query in draw order; a candidate is rejected when it lies in an inflated obstacle
//                     (max(A x - b) < 1e-3, :467-471) or in a known set (max(a_set x - b_set) < 1e-3, :472-476);
//                     out: the first accepted candidate.  One CTA per query, one warp per candidate in flight.
//   k_dedupe_dist     the duplicate-set test (:505-512): min over the query's graph nodes of
//                     ||Q - Q_v||_F + ||p - p_v||.  One warp per new set.
//   k_shortest_path   nx.shortest_path(inter_graph, 0, 1, weight) (:434): Dijkstra on a small weighted graph in
//                     CSR form, one warp per graph (lanes over nodes for the argmin, over edges for the relaxation).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_sample_filter(SceneView sc_all, const double* __restrict__ cand, int C,
                                                       const double* __restrict__ A, const double* __restrict__ b,
                                                       const int* __restrict__ m, int m_max,
                                                       const int* __restrict__ set_off,
                                                       const int* __restrict__ set_cnt, int* __restrict__ first_ok,
                                                       unsigned char* __restrict__ flags) {
  const SceneView sc = scene_of_item(sc_all, blockIdx.x);
  __shared__ int s_first;
  const int q = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned full = 0xffffffffu;
  if (threadIdx.x == 0) s_first = 0x7fffffff;
  __syncthreads();
  // known sets of query q: rows set_off[q] .. set_off[q+1]-1, or (set_cnt given) set_off[q] .. set_off[q]+set_cnt[q]-1
  const int s0 = set_off ? set_off[q] : 0, s1 = set_off ? (set_cnt ? s0 + set_cnt[q] : set_off[q + 1]) : 0;
  for (int base = 0; base < C; base += 4) {
    const int c = base + warp;
    if (c < C) {
      const double x0 = cand[((size_t)q * C + c) * 3], x1 = cand[((size_t)q * C + c) * 3 + 1],
                   x2 = cand[((size_t)q * C + c) * 3 + 2];
      bool coll = false, safe = false;
      for (int j = lane; j < sc.n; j += 32) {
        double lb[3], ub[3];
        load_box(sc, j, lb, ub);
        // rows +-e_k of the inflated box: A x - b = x_k - ub_k, lb_k - x_k (padded rows give -10)
        double v = fmax(fmax(fmax(x0 - ub[0], lb[0] - x0), fmax(x1 - ub[1], lb[1] - x1)), fmax(x2 - ub[2], lb[2] - x2));
        if (sc.rows) {
          // general polytope: the reference's test is max(A x - b) < 1e-3 over the obstacle's own rows (:467-471).
          // No bounding-box gate: near a sharp vertex or edge that region reaches 1e-3 / sin(theta / 2) beyond the
          // polytope, i.e. outside any fixed growth of the vertex bounding box
          const double* r4 = sc.rows + (size_t)j * BP_OBS_ROWS * 4;
          v = -10.0;                                // the padded rows' A x - b (only matters for an obstacle without rows)
          for (int r = 0; r < sc.nrows[j]; ++r)
            v = fmax(v, (__ldg(r4 + 4 * r) * x0 + __ldg(r4 + 4 * r + 1) * x1 + __ldg(r4 + 4 * r + 2) * x2) - __ldg(r4 + 4 * r + 3));
        }
        coll |= v < 1e-3;
      }
      for (int t = s0 + lane; t < s1; t += 32) {
        const double* At = A + (size_t)t * m_max * 3;
        const double* bt = b + (size_t)t * m_max;
        double v = -BP_INF;
        for (int r = 0; r < m[t]; ++r) v = fmax(v, (At[3 * r] * x0 + At[3 * r + 1] * x1 + At[3 * r + 2] * x2) - bt[r]);
        safe |= (m[t] > 0) && (v < 1e-3);
      }
      coll = __any_sync(full, coll);
      safe = __any_sync(full, safe);
      if (lane == 0) {
        if (flags) flags[(size_t)q * C + c] = (unsigned char)((coll ? 1 : 0) | (safe ? 2 : 0));
        if (!coll && !safe) atomicMin(&s_first, c);
      }
    }
    __syncthreads();
    const int found = s_first;
    __syncthreads();                                 // nobody updates s_first for the next group before all have read it
    if (!flags && found < 0x7fffffff) break;         // (with flags every candidate is classified)
  }
  if (threadIdx.x == 0) first_ok[q] = s_first < 0x7fffffff ? s_first : -1;
}

__global__ void __launch_bounds__(32) k_dedupe_dist(const double* __restrict__ q_new, const double* __restrict__ p_new,
                                                    const double* __restrict__ q_nodes,
                                                    const double* __restrict__ p_nodes,
                                                    const int* __restrict__ node_off,
                                                    const int* __restrict__ node_cnt, double* __restrict__ dmin,
                                                    int* __restrict__ argmin) {
  const int i = blockIdx.x, lane = threadIdx.x;
  double best = BP_INF;
  int bidx = 0x7fffffff;
  const int v_end = node_cnt ? node_off[i] + node_cnt[i] : node_off[i + 1];
  for (int v = node_off[i] + lane; v < v_end; v += 32) {
    double sq = 0.0, sp = 0.0;
#pragma unroll
    for (int k = 0; k < 9; ++k) { const double d = q_new[(size_t)i * 9 + k] - q_nodes[(size_t)v * 9 + k]; sq += d * d; }
#pragma unroll
    for (int k = 0; k < 3; ++k) { const double d = p_new[(size_t)i * 3 + k] - p_nodes[(size_t)v * 3 + k]; sp += d * d; }
    const double d = sqrt(sq) + sqrt(sp);
    if (d < best) { best = d; bidx = v - node_off[i]; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
    if (ov < best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
  }
  if (lane == 0) { dmin[i] = best; if (argmin) argmin[i] = bidx < 0x7fffffff ? bidx : -1; }
}

#define BP_SP_MAX_NODES 1024
__global__ void __launch_bounds__(32) k_shortest_path(const int* __restrict__ node_off, const int* __restrict__ edge_off,
                                                      const int* __restrict__ edge_dst,
                                                      const double* __restrict__ edge_w, const int* __restrict__ src,
                                                      const int* __restrict__ dst, int max_len,
                                                      int* __restrict__ path, int* __restrict__ path_len,
                                                      double* __restrict__ cost) {
  __shared__ double s_d[BP_SP_MAX_NODES];
  __shared__ int s_pred[BP_SP_MAX_NODES];
  __shared__ unsigned char s_done[BP_SP_MAX_NODES];
  const int g = blockIdx.x, lane = threadIdx.x;
  const unsigned full = 0xffffffffu;
  const int n0 = node_off[g], n = node_off[g + 1] - n0;        // nodes of this graph are n0 .. n0 + n - 1
  const int* eoff = edge_off + n0;                              // CSR rows of the graph's nodes (global edge ids)
  for (int v = lane; v < n; v += 32) { s_d[v] = BP_INF; s_pred[v] = -1; s_done[v] = 0; }
  __syncwarp();
  const int a = src[g], z = dst[g];
  int len = -1;
  if (n > 0 && n <= BP_SP_MAX_NODES && a >= 0 && a < n && z >= 0 && z < n) {
    if (lane == 0) s_d[a] = 0.0;
    __syncwarp();
    for (int it = 0; it < n; ++it) {
      double best = BP_INF;
      int u = 0x7fffffff;
      for (int v = lane; v < n; v += 32)
        if (!s_done[v] && s_d[v] < best) { best = s_d[v]; u = v; }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(full, best, off);
        const int ou = __shfl_xor_sync(full, u, off);
        if (ov < best || (ov == best && ou < u)) { best = ov; u = ou; }
      }
      if (!(best < BP_INF)) break;                              // the rest is unreachable
      __syncwarp();                                             // every lane's scan of s_done precedes the write
      if (lane == 0) s_done[u] = 1;
      if (u == z) break;
      __syncwarp();
      for (int e = eoff[u] + lane; e < eoff[u + 1]; e += 32) {
        const int v = edge_dst[e];
        const double nd = best + edge_w[e];
        if (!s_done[v] && nd < s_d[v]) { s_d[v] = nd; s_pred[v] = u; }   // distinct v per edge of u (simple graph)
      }
      __syncwarp();
    }
    __syncwarp();
    if (s_d[z] < BP_INF) {
      len = 1;
      for (int v = z; v != a; v = s_pred[v]) ++len;
      if (len <= max_len && lane == 0) {
        int v = z;
        for (int k = len - 1; k >= 0; --k) { path[(size_t)g * max_len + k] = v; v = s_pred[v]; }
      }
    }
  }
  if (lane == 0) {
    path_len[g] = len;
    cost[g] = len > 0 ? s_d[z] : BP_INF;
  }
}

// ---------------------------------------------------------------------------
// Multi-GPU exchange by peer stores over NVLink (SURVEY 8e): instead of packing the sets, calling an NCCL
// all-gather and unpacking, the owner writes every set straight into the global tables of EVERY rank (its own
// included) through the peers' mapped addresses -- A[S,m_max,3], b[S,m_max], m[S] and the bounding boxes
// [S,6] at row slot0 + s.  The adjacency row block goes out the same way.  peer_base[r] is the base address
// of rank r's symmetric allocation (same layout on every rank), off_* the byte offsets of the tables in it.
// One cross-rank barrier (the symmetric-memory signal pads) follows each scatter; nothing is staged or copied.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_scatter_sets_peers(const double* __restrict__ A, const double* __restrict__ b,
                                                            const int* __restrict__ m,
                                                            const double* __restrict__ aabb, int m_max, int slot0,
                                                            const unsigned long long* __restrict__ peer_base,
                                                            int world, size_t off_A, size_t off_b, size_t off_m,
                                                            size_t off_aabb) {
  const int s = blockIdx.x, g = slot0 + s, tid = threadIdx.x;
  const double* As = A + (size_t)s * m_max * 3;
  const double* bs = b + (size_t)s * m_max;
  for (int r = 0; r < world; ++r) {
    char* base = (char*)peer_base[r];
    double* Ad = (double*)(base + off_A) + (size_t)g * m_max * 3;
    double* bd = (double*)(base + off_b) + (size_t)g * m_max;
    for (int e = tid; e < 3 * m_max; e += blockDim.x) Ad[e] = As[e];
    for (int e = tid; e < m_max; e += blockDim.x) bd[e] = bs[e];
    if (tid < 6) ((double*)(base + off_aabb))[(size_t)g * 6 + tid] = aabb[(size_t)s * 6 + tid];
    if (tid == 6) ((int*)(base + off_m))[g] = m[s];
  }
}

__global__ void __launch_bounds__(256) k_scatter_rows_peers(const unsigned int* __restrict__ rows_local, int rows,
                                                            int words, int row0,
                                                            const unsigned long long* __restrict__ peer_base,
                                                            int world, size_t off_bits) {
  const size_t n = (size_t)rows * words;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const unsigned int v = rows_local[e];
    for (int r = 0; r < world; ++r) ((unsigned int*)((char*)peer_base[r] + off_bits))[(size_t)row0 * words + e] = v;
  }
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
template <bool POSE, bool JAC>
static int launch_fk(const double* q, int B, double* p_ee, double* p_col, double* T_ee, double* jac, int use_tma,
                     cudaStream_t stream) {
  const size_t smem = sizeof(double) * FK_T * (7 + 3 + 21 + (POSE ? 16 : 0) + (JAC ? 42 : 0));
  if (smem > 48 * 1024)
    BP_CUDA(cudaFuncSetAttribute((const void*)k_fk<POSE, JAC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_fk<POSE, JAC><<<(B + FK_T - 1) / FK_T, FK_T, smem, stream>>>(q, B, p_ee, p_col, T_ee, jac, use_tma);
  BP_CUDA(cudaGetLastError());
  return 0;
}

// closest points are cached in shared memory while dist[N] + y[3][N] stays within 96 KB per CTA
static int poly_cache_y(int n) { return (size_t)n * 32 <= 96 * 1024; }
// polytope scenes: dist[N] (+ y[3][N] while that fits); box scenes: key2[N] + the shell (poly_pass_shell)
static size_t poly_smem_bytes(int n, bool polytopes) {
  if (n < 1) n = 1;
  if (polytopes) return sizeof(double) * (size_t)n * (poly_cache_y(n) ? 4 : 1);
  return sizeof(double) * (size_t)((n + 1) & ~1) + sizeof(ShellMem);
}
// k_poly_point on box scenes: the shell form while key table + shell fit next to 1 KB of static shared memory
static bool poly_point_shell(int n) { return poly_smem_bytes(n, false) + 1024 <= 227 * 1024; }
static size_t poly_point_smem_bytes(int n, bool polytopes) {
  if (polytopes || poly_point_shell(n)) return poly_smem_bytes(n, polytopes);
  return sizeof(double) * (size_t)n;
}
// fused per-seed kernel for small / medium scenes; BPGEO_FUSED=0 forces the launch sequence
#define BP_POLY_SCENE_MAX 16384               // polytope scenes: obstacles per scene (one alive bit per thread and entry)
static bool use_fused_iris(int n) {
  static int env = -1;
  if (env < 0) {
    const char* e = getenv("BPGEO_FUSED");
    env = (e && e[0] == '0') ? 0 : 1;
  }
  return env == 1 && n <= 16384;            // 128 threads x 2 words of alive bits
}
static int poly_threads(int n) { return n <= 256 ? 128 : (n <= 4096 ? 256 : 512); }

static int set_dyn_smem(const void* fn, size_t bytes) {
  // the opt-in limit (227 KB on sm_100a) covers the kernel's static shared memory as well
  cudaFuncAttributes fa;
  BP_CUDA(cudaFuncGetAttributes(&fa, fn));
  int dev = 0, optin = 0;
  BP_CUDA(cudaGetDevice(&dev));
  BP_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (bytes + fa.sharedSizeBytes > (size_t)optin) {
    snprintf(g_err, sizeof(g_err),
             "scene too large for the shared-memory distance table (%zu B dynamic + %zu B static > %d B per CTA; "
             "N <= %zu)", bytes, (size_t)fa.sharedSizeBytes, optin, ((size_t)optin - fa.sharedSizeBytes) / sizeof(double));
    return 1;
  }
  // (the 48 KB default limit counts static + dynamic shared memory)
  if (bytes + fa.sharedSizeBytes > 48 * 1024)
    BP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

// ---------------------------------------------------------------------------
// Device ingest of a scene batch (bp_scene_update_batch / bp_scene_update_polytopes_batch): the new obstacles arrive
// in one staging copy and are written into the resident layout by the kernels below, with the host arithmetic of
// scene_upload / bp_scene_create_polytopes, so that the updated batch holds the bits of a freshly created one.
// ---------------------------------------------------------------------------
// boxes [total,6] (lb | ub) -> the six columns lb - inflate | ub + inflate of stride cap, zeros in [total, cap);
// offsets [n_seg+1] -> seg_off
__global__ void __launch_bounds__(256) k_scene_ingest_boxes(const double* __restrict__ boxes, int total, int cap,
                                                            double inflate, double* __restrict__ cols,
                                                            const int* __restrict__ offsets, int n_seg,
                                                            int* __restrict__ seg_off) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_seg + 1) seg_off[j] = offsets[j];
  if (j >= cap) return;
  const bool real = j < total;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    cols[(size_t)k * cap + j] = real ? boxes[6 * (size_t)j + k] - inflate : 0.0;
    cols[(size_t)(3 + k) * cap + j] = real ? boxes[6 * (size_t)j + 3 + k] + inflate : 0.0;
  }
}

// the vertices of every obstacle (rows [total,15,4], nrows [total]) into V [total,vmax,3] / nv [total]; flags[0]
// receives the smallest 2 j + (1: too many vertices, 0: not a polytope) over the failing obstacles, flags[1] the
// largest vertex count
__global__ void __launch_bounds__(128) k_scene_enum_vertices(const double* __restrict__ rows,
                                                             const int* __restrict__ nrows, int vmax,
                                                             double* __restrict__ V, int* __restrict__ nv,
                                                             int* __restrict__ flags) {
  __shared__ double sA[BP_OBS_ROWS * 3], sb[BP_OBS_ROWS];
  const int j = blockIdx.x, tid = threadIdx.x;
  const int ms = nrows[j];
  const double* r4 = rows + (size_t)j * BP_OBS_ROWS * 4;
  for (int e = tid; e < ms * 3; e += 128) sA[e] = r4[4 * (e / 3) + e % 3];
  for (int e = tid; e < ms; e += 128) sb[e] = r4[4 * e + 3];
  const int stt = polytope_vertices_cta(sA, sb, ms, vmax, V + (size_t)j * vmax * 3, nv + j);
  if (tid == 0) {
    if (stt != BP_OK) atomicMin(&flags[0], 2 * j + (stt == BP_ROW_OVERFLOW ? 1 : 0));
    else atomicMax(&flags[1], nv[j]);
  }
}

// one warp per obstacle: rows / nrows copied, the vertices (src stride vmax_in) re-strided to vmax with zeros after
// the last one, nverts, and the bounding box of the vertices (the min / max loop of bp_scene_create_polytopes, then
// scene_upload's "- inflate" / "+ inflate" with inflate = 0) into the columns; zeros in [total, cap); seg_off
__global__ void __launch_bounds__(256) k_scene_ingest_polytopes(
    const double* __restrict__ rows_in, const int* __restrict__ nrows_in, const double* __restrict__ verts_in,
    const int* __restrict__ nverts_in, int vmax_in, int total, int vmax, int cap, double inflate,
    double* __restrict__ rows, int* __restrict__ nrows, double* __restrict__ verts, int* __restrict__ nverts,
    double* __restrict__ cols, const int* __restrict__ offsets, int n_seg, int* __restrict__ seg_off) {
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (blockIdx.x == 0)
    for (int e = threadIdx.x; e < n_seg + 1; e += blockDim.x) seg_off[e] = offsets[e];
  if (j >= cap) return;
  if (j >= total) {
    if (lane < 6) cols[(size_t)lane * cap + j] = 0.0;
    return;
  }
  for (int e = lane; e < BP_OBS_ROWS * 4; e += 32) rows[(size_t)j * BP_OBS_ROWS * 4 + e] = rows_in[(size_t)j * BP_OBS_ROWS * 4 + e];
  const int nv = nverts_in[j];
  const double* src = verts_in + (size_t)j * vmax_in * 3;
  for (int e = lane; e < vmax * 3; e += 32) verts[(size_t)j * vmax * 3 + e] = e < nv * 3 ? src[e] : 0.0;
  if (lane == 0) { nrows[j] = nrows_in[j]; nverts[j] = nv; }
  if (lane < 3) {
    double lo = BP_INF, hi = -BP_INF;
    for (int t = 0; t < nv; ++t) {
      const double v = src[3 * t + lane];
      if (v < lo) lo = v;
      if (v > hi) hi = v;
    }
    cols[(size_t)lane * cap + j] = lo - inflate;
    cols[(size_t)(3 + lane) * cap + j] = hi + inflate;
  }
}

extern "C" {

int bpgeo_abi_version(void) { return BPGEO_ABI_VERSION; }
#ifdef BPGEO_PROFILE
int bp_prof_read_mvie(long long* host_out, int n_seeds, int reset) {
  BP_CUDA(cudaDeviceSynchronize());
  BP_CUDA(cudaMemcpyFromSymbol(host_out, g_prof_mvie, sizeof(long long) * 8 * (size_t)n_seeds));
  if (reset) {
    void* ptr = nullptr;
    BP_CUDA(cudaGetSymbolAddress(&ptr, g_prof_mvie));
    BP_CUDA(cudaMemset(ptr, 0, sizeof(g_prof_mvie)));
  }
  return 0;
}
int bp_prof_read_pair(long long* host_out, int reset) {
  BP_CUDA(cudaDeviceSynchronize());
  BP_CUDA(cudaMemcpyFromSymbol(host_out, g_prof_pair, sizeof(g_prof_pair)));
  if (reset) {
    void* ptr = nullptr;
    BP_CUDA(cudaGetSymbolAddress(&ptr, g_prof_pair));
    BP_CUDA(cudaMemset(ptr, 0, sizeof(g_prof_pair)));
  }
  return 0;
}
int bp_prof_read_poly(long long* host_out, int n_seeds, int reset) {
  BP_CUDA(cudaDeviceSynchronize());
  BP_CUDA(cudaMemcpyFromSymbol(host_out, g_prof_poly, sizeof(long long) * 8 * (size_t)n_seeds));
  if (reset) {
    void* ptr = nullptr;
    BP_CUDA(cudaGetSymbolAddress(&ptr, g_prof_poly));
    BP_CUDA(cudaMemset(ptr, 0, sizeof(g_prof_poly)));
  }
  return 0;
}
int bp_prof_read(long long* host_out, int n_seeds, int reset) {
  BP_CUDA(cudaDeviceSynchronize());
  BP_CUDA(cudaMemcpyFromSymbol(host_out, g_prof, sizeof(long long) * 4 * (size_t)n_seeds));
  if (reset) {
    void* ptr = nullptr;
    BP_CUDA(cudaGetSymbolAddress(&ptr, g_prof));
    BP_CUDA(cudaMemset(ptr, 0, sizeof(g_prof)));
  }
  return 0;
}
#endif
const char* bp_last_error_string(void) { return g_err; }

static int set_seg_off_host(bp_scene* sc, const int* offsets_host) {
  if (!sc->seg_off_host) sc->seg_off_host = (int*)malloc(sizeof(int) * (size_t)(sc->n_seg + 1));
  if (!sc->seg_off_host) return bp_fail("out of host memory");
  memcpy(sc->seg_off_host, offsets_host, sizeof(int) * (size_t)(sc->n_seg + 1));
  return 0;
}

static int scene_upload(bp_scene* sc, const double* boxes_host, int n, double inflate, cudaStream_t stream) {
  if (n > sc->cap) {
    if (sc->cols) BP_CUDA(cudaFree(sc->cols));
    sc->cols = nullptr;
    sc->cap = ((n + 31) / 32) * 32;
    BP_CUDA(cudaMalloc(&sc->cols, sizeof(double) * 6 * (size_t)sc->cap));
  }
  sc->n = n;
  sc->inflate = inflate;
  if (n == 0) return 0;
  double* tmp = (double*)malloc(sizeof(double) * 6 * (size_t)sc->cap);
  if (!tmp) return bp_fail("out of host memory");
  memset(tmp, 0, sizeof(double) * 6 * (size_t)sc->cap);
  for (int j = 0; j < n; ++j)
    for (int k = 0; k < 3; ++k) {
      tmp[(size_t)k * sc->cap + j] = boxes_host[6 * j + k] - inflate;          // -lb + inflate  (:141)
      tmp[(size_t)(3 + k) * sc->cap + j] = boxes_host[6 * j + 3 + k] + inflate;
    }
  cudaError_t e = cudaMemcpyAsync(sc->cols, tmp, sizeof(double) * 6 * (size_t)sc->cap, cudaMemcpyHostToDevice, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  free(tmp);
  if (e != cudaSuccess) return bp_fail("scene upload", e);
  return 0;
}

int bp_scene_create(const double* boxes_host, int n, double inflate, bp_scene** out) {
  if (!out || n < 0 || (n > 0 && !boxes_host)) return bp_fail("bp_scene_create: bad arguments");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return bp_fail("bp_scene_create: no CUDA device (libbpgeo has no CPU fallback)", e);
  bp_scene* sc = (bp_scene*)calloc(1, sizeof(bp_scene));
  if (!sc) return bp_fail("out of host memory");
  int rc = scene_upload(sc, boxes_host, n, inflate, 0);
  if (rc) { free(sc); return rc; }
  *out = sc;
  return 0;
}

int bp_scene_create_batch(const double* boxes_host, const int* offsets_host, int n_scenes, double inflate,
                          bp_scene** out) {
  if (!out || n_scenes < 1 || !offsets_host || offsets_host[0] != 0) return bp_fail("bp_scene_create_batch: bad arguments");
  int n_max = 0;
  for (int k = 0; k < n_scenes; ++k) {
    const int nk = offsets_host[k + 1] - offsets_host[k];
    if (nk < 0) return bp_fail("bp_scene_create_batch: offsets must be non-decreasing");
    n_max = nk > n_max ? nk : n_max;
  }
  const int total = offsets_host[n_scenes];
  bp_scene* sc = nullptr;
  int rc = bp_scene_create(boxes_host, total, inflate, &sc);
  if (rc) return rc;
  sc->n = n_max;                                  // sizes shared memory / picks the kernel variant
  sc->n_seg = n_scenes;
  cudaError_t e = cudaMalloc(&sc->seg_off, sizeof(int) * (size_t)(n_scenes + 1));
  if (e == cudaSuccess)
    e = cudaMemcpy(sc->seg_off, offsets_host, sizeof(int) * (size_t)(n_scenes + 1), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { bp_scene_destroy(sc); return bp_fail("bp_scene_create_batch", e); }
  if (set_seg_off_host(sc, offsets_host)) { bp_scene_destroy(sc); return 1; }
  *out = sc;
  return 0;
}

int bp_scene_create_polytopes(const double* rows_host, const int* nrows_host, const double* verts_host,
                              const int* nverts_host, int n, int vmax, bp_scene** out) {
  if (!out || n < 1 || vmax < 1 || !rows_host || !nrows_host || !verts_host || !nverts_host)
    return bp_fail("bp_scene_create_polytopes: bad arguments");
  // bounding boxes from the vertices: the cheap lower bounds of the lazy closest-point pass
  double* boxes = (double*)malloc(sizeof(double) * 6 * (size_t)n);
  if (!boxes) return bp_fail("out of host memory");
  for (int j = 0; j < n; ++j) {
    if (nrows_host[j] < 1 || nrows_host[j] > BP_OBS_ROWS || nverts_host[j] < 1 || nverts_host[j] > vmax) {
      free(boxes);
      return bp_fail("bp_scene_create_polytopes: an obstacle needs 1..15 rows and 1..vmax vertices");
    }
    for (int k = 0; k < 3; ++k) { boxes[6 * j + k] = BP_INF; boxes[6 * j + 3 + k] = -BP_INF; }
    for (int t = 0; t < nverts_host[j]; ++t)
      for (int k = 0; k < 3; ++k) {
        const double v = verts_host[((size_t)j * vmax + t) * 3 + k];
        if (v < boxes[6 * j + k]) boxes[6 * j + k] = v;
        if (v > boxes[6 * j + 3 + k]) boxes[6 * j + 3 + k] = v;
      }
  }
  bp_scene* sc = nullptr;
  int rc = bp_scene_create(boxes, n, 0.0, &sc);
  free(boxes);
  if (rc) return rc;
  cudaError_t e = cudaMalloc(&sc->rows, sizeof(double) * (size_t)n * BP_OBS_ROWS * 4);
  if (e == cudaSuccess) e = cudaMalloc(&sc->nrows, sizeof(int) * (size_t)n);
  if (e == cudaSuccess) e = cudaMalloc(&sc->verts, sizeof(double) * (size_t)n * vmax * 3);
  if (e == cudaSuccess) e = cudaMalloc(&sc->nverts, sizeof(int) * (size_t)n);
  if (e == cudaSuccess) e = cudaMemcpy(sc->rows, rows_host, sizeof(double) * (size_t)n * BP_OBS_ROWS * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(sc->nrows, nrows_host, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(sc->verts, verts_host, sizeof(double) * (size_t)n * vmax * 3, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(sc->nverts, nverts_host, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice);
  sc->vmax = vmax;
  sc->pcap = n;
  sc->vcap = (size_t)n * vmax * 3;
  if (e != cudaSuccess) { bp_scene_destroy(sc); return bp_fail("bp_scene_create_polytopes", e); }
  *out = sc;
  return 0;
}

int bp_scene_create_polytopes_batch(const double* rows_host, const int* nrows_host, const double* verts_host,
                                    const int* nverts_host, const int* offsets_host, int n_scenes, int vmax,
                                    bp_scene** out) {
  if (!out || n_scenes < 1 || !offsets_host || offsets_host[0] != 0)
    return bp_fail("bp_scene_create_polytopes_batch: bad arguments");
  int n_max = 0;
  for (int k = 0; k < n_scenes; ++k) {
    const int nk = offsets_host[k + 1] - offsets_host[k];
    if (nk < 0) return bp_fail("bp_scene_create_polytopes_batch: offsets must be non-decreasing");
    n_max = nk > n_max ? nk : n_max;
  }
  bp_scene* sc = nullptr;
  int rc = bp_scene_create_polytopes(rows_host, nrows_host, verts_host, nverts_host, offsets_host[n_scenes], vmax, &sc);
  if (rc) return rc;
  sc->n = n_max;                                  // sizes shared memory / picks the kernel variant
  sc->n_seg = n_scenes;
  cudaError_t e = cudaMalloc(&sc->seg_off, sizeof(int) * (size_t)(n_scenes + 1));
  if (e == cudaSuccess)
    e = cudaMemcpy(sc->seg_off, offsets_host, sizeof(int) * (size_t)(n_scenes + 1), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { bp_scene_destroy(sc); return bp_fail("bp_scene_create_polytopes_batch", e); }
  if (set_seg_off_host(sc, offsets_host)) { bp_scene_destroy(sc); return 1; }
  *out = sc;
  return 0;
}

int bp_scene_update(bp_scene* scene, const double* boxes_host, int n, double inflate, void* stream) {
  if (scene && scene->seg_off) return bp_fail("bp_scene_update: not supported for scene batches");
  if (scene && scene->rows) return bp_fail("bp_scene_update: not supported for polytope scenes (create a new one)");
  if (!scene || n < 0 || (n > 0 && !boxes_host)) return bp_fail("bp_scene_update: bad arguments");
  return scene_upload(scene, boxes_host, n, inflate, (cudaStream_t)stream);
}

// checks of a batch update: the scene is a batch of the given kind and of n_scenes scenes, the offsets start at 0
// and do not decrease; returns the largest scene size, or -1 (g_err set)
static int update_check(const bp_scene* sc, const int* offsets_host, int n_scenes, bool polytopes, const char* fn) {
  if (!sc || !offsets_host || n_scenes < 1 || offsets_host[0] != 0) {
    snprintf(g_err, sizeof(g_err), "%s: bad arguments", fn);
    return -1;
  }
  if (!sc->seg_off) {
    snprintf(g_err, sizeof(g_err), "%s: not a scene batch", fn);
    return -1;
  }
  if ((sc->rows != nullptr) != polytopes) {
    snprintf(g_err, sizeof(g_err), "%s: the scene batch holds %s (use %s)", fn, sc->rows ? "polytopes" : "boxes",
             sc->rows ? "bp_scene_update_polytopes_batch" : "bp_scene_update_batch");
    return -1;
  }
  if (n_scenes != sc->n_seg) {
    snprintf(g_err, sizeof(g_err), "%s: %d scenes for a batch of %d", fn, n_scenes, sc->n_seg);
    return -1;
  }
  int n_max = 0;
  for (int k = 0; k < n_scenes; ++k) {
    const int nk = offsets_host[k + 1] - offsets_host[k];
    if (nk < 0) {
      snprintf(g_err, sizeof(g_err), "%s: offsets must be non-decreasing", fn);
      return -1;
    }
    n_max = nk > n_max ? nk : n_max;
  }
  return n_max;
}

// the scene of obstacle j of a batch
static int scene_of_obstacle(const int* offsets_host, int j) {
  int k = 0;
  while (offsets_host[k + 1] <= j) ++k;
  return k;
}

static size_t stage_align(size_t b) { return (b + 255) & ~(size_t)255; }

// grow the update staging to hbytes pinned host / dbytes device bytes (the new buffer before the old one is released)
static int stage_reserve(bp_scene* sc, size_t hbytes, size_t dbytes) {
  if (hbytes > sc->stage_h_cap) {
    void* p = nullptr;
    const size_t cap = hbytes + hbytes / 4;
    BP_CUDA(cudaMallocHost(&p, cap));
    if (sc->stage_h) cudaFreeHost(sc->stage_h);
    sc->stage_h = p;
    sc->stage_h_cap = cap;
  }
  if (dbytes > sc->stage_d_cap) {
    void* p = nullptr;
    const size_t cap = dbytes + dbytes / 4;
    BP_CUDA(cudaMalloc(&p, cap));
    if (sc->stage_d) cudaFree(sc->stage_d);
    sc->stage_d = p;
    sc->stage_d_cap = cap;
  }
  return 0;
}

int bp_scene_update_batch(bp_scene* scene, const double* boxes_host, const int* offsets_host, int n_scenes,
                          double inflate, void* stream) {
  const int n_max = update_check(scene, offsets_host, n_scenes, false, "bp_scene_update_batch");
  if (n_max < 0) return 1;
  const int total = offsets_host[n_scenes];
  if (total > 0 && !boxes_host) return bp_fail("bp_scene_update_batch: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  // staging: boxes [total,6] | offsets [n_scenes+1]
  const size_t o_off = stage_align(sizeof(double) * 6 * (size_t)total);
  const size_t bytes = o_off + sizeof(int) * (size_t)(n_scenes + 1);
  if (stage_reserve(scene, bytes, bytes)) return 1;
  int new_cap = scene->cap;
  double* cols = scene->cols;
  if (total > scene->cap) {
    new_cap = ((total + 31) / 32) * 32;
    BP_CUDA(cudaMalloc(&cols, sizeof(double) * 6 * (size_t)new_cap));
  }
  char* h = (char*)scene->stage_h;
  const char* d = (const char*)scene->stage_d;
  if (total > 0) memcpy(h, boxes_host, sizeof(double) * 6 * (size_t)total);
  memcpy(h + o_off, offsets_host, sizeof(int) * (size_t)(n_scenes + 1));
  cudaError_t e = cudaMemcpyAsync(scene->stage_d, h, bytes, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    const int items = new_cap > n_scenes + 1 ? new_cap : n_scenes + 1;
    k_scene_ingest_boxes<<<(items + 255) / 256, 256, 0, st>>>((const double*)d, total, new_cap, inflate, cols,
                                                             (const int*)(d + o_off), n_scenes, scene->seg_off);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);      // (the pinned staging is reused by the next update)
  if (e != cudaSuccess) {
    if (cols != scene->cols) cudaFree(cols);
    return bp_fail("bp_scene_update_batch", e);
  }
  if (cols != scene->cols) {
    if (scene->cols) cudaFree(scene->cols);
    scene->cols = cols;
    scene->cap = new_cap;
  }
  scene->n = n_max;
  scene->inflate = inflate;
  memcpy(scene->seg_off_host, offsets_host, sizeof(int) * (size_t)(n_scenes + 1));
  return 0;
}

#define BP_ENUM_VMAX 64                       // vertices per obstacle enumerated by bp_scene_update_polytopes_batch

int bp_scene_update_polytopes_batch(bp_scene* scene, const double* rows_host, const int* nrows_host,
                                    const double* verts_host, const int* nverts_host, const int* offsets_host,
                                    int n_scenes, int vmax, void* stream) {
  const char* fn = "bp_scene_update_polytopes_batch";
  const int n_max = update_check(scene, offsets_host, n_scenes, true, fn);
  if (n_max < 0) return 1;
  const int total = offsets_host[n_scenes];
  const bool given = verts_host != nullptr;
  if (!rows_host || !nrows_host || (given && (!nverts_host || vmax < 1)))
    return bp_fail("bp_scene_update_polytopes_batch: bad arguments");
  if (total < 1) return bp_fail("bp_scene_update_polytopes_batch: a polytope scene batch needs at least one obstacle");
  int vmax_new = 0;
  for (int j = 0; j < total; ++j) {
    if (nrows_host[j] < 1 || nrows_host[j] > BP_OBS_ROWS || (given && (nverts_host[j] < 1 || nverts_host[j] > vmax))) {
      const int k = scene_of_obstacle(offsets_host, j);
      snprintf(g_err, sizeof(g_err), "%s: scene %d, obstacle %d needs 1..15 rows%s", fn, k, j - offsets_host[k],
               given ? " and 1..vmax vertices" : "");
      return 1;
    }
    if (given && nverts_host[j] > vmax_new) vmax_new = nverts_host[j];
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int vin = given ? vmax : BP_ENUM_VMAX;           // vertex stride of the ingest's source
  // staging, host and device: rows [total,15,4] | nrows [total] | offsets [n_scenes+1] | flags [2] | (given)
  // verts [total,vmax,3] | nverts [total]; device only, when enumerating: V [total,64,3] | nv [total]
  const size_t o_nrows = stage_align(sizeof(double) * (size_t)total * BP_OBS_ROWS * 4);
  const size_t o_off = o_nrows + stage_align(sizeof(int) * (size_t)total);
  const size_t o_flags = o_off + stage_align(sizeof(int) * (size_t)(n_scenes + 1));
  const size_t o_verts = o_flags + stage_align(sizeof(int) * 2);
  const size_t o_nverts = o_verts + stage_align(sizeof(double) * (size_t)total * vin * 3);
  const size_t hbytes = given ? o_nverts + sizeof(int) * (size_t)total : o_verts;
  const size_t dbytes = o_nverts + sizeof(int) * (size_t)total;
  if (stage_reserve(scene, hbytes, dbytes)) return 1;
  char* h = (char*)scene->stage_h;
  char* d = (char*)scene->stage_d;
  memcpy(h, rows_host, sizeof(double) * (size_t)total * BP_OBS_ROWS * 4);
  memcpy(h + o_nrows, nrows_host, sizeof(int) * (size_t)total);
  memcpy(h + o_off, offsets_host, sizeof(int) * (size_t)(n_scenes + 1));
  int* flags_h = (int*)(h + o_flags);
  flags_h[0] = 0x7fffffff;
  flags_h[1] = 0;
  if (given) {
    memcpy(h + o_verts, verts_host, sizeof(double) * (size_t)total * vmax * 3);
    memcpy(h + o_nverts, nverts_host, sizeof(int) * (size_t)total);
  }
  BP_CUDA(cudaMemcpyAsync(d, h, hbytes, cudaMemcpyHostToDevice, st));
  if (!given) {
    // enumerate into the staging and commit only when every obstacle is a polytope of at most 64 vertices
    k_scene_enum_vertices<<<total, 128, 0, st>>>((const double*)d, (const int*)(d + o_nrows), BP_ENUM_VMAX,
                                                 (double*)(d + o_verts), (int*)(d + o_nverts), (int*)(d + o_flags));
    BP_CUDA(cudaGetLastError());
    BP_CUDA(cudaMemcpyAsync(flags_h, d + o_flags, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
    BP_CUDA(cudaStreamSynchronize(st));
    if (flags_h[0] != 0x7fffffff) {
      const int j = flags_h[0] / 2, k = scene_of_obstacle(offsets_host, j);
      if (flags_h[0] & 1)
        snprintf(g_err, sizeof(g_err), "%s: scene %d, obstacle %d has more than %d vertices", fn, k, j - offsets_host[k],
                 BP_ENUM_VMAX);
      else
        snprintf(g_err, sizeof(g_err), "%s: scene %d, obstacle %d: Polyhedron is not a polytope", fn, k,
                 j - offsets_host[k]);
      return 1;
    }
    vmax_new = flags_h[1];
  }
  // buffers that have to grow: all allocated before anything is released
  double *rows = scene->rows, *verts = scene->verts, *cols = scene->cols;
  int *nrows = scene->nrows, *nverts = scene->nverts;
  const int pcap = total > scene->pcap ? total : scene->pcap;
  const size_t vneed = (size_t)total * vmax_new * 3, vcap = vneed > scene->vcap ? vneed : scene->vcap;
  const int cap = total > scene->cap ? ((total + 31) / 32) * 32 : scene->cap;
  cudaError_t e = cudaSuccess;
  if (pcap != scene->pcap) {
    rows = nullptr; nrows = nullptr; nverts = nullptr;
    e = cudaMalloc(&rows, sizeof(double) * (size_t)pcap * BP_OBS_ROWS * 4);
    if (e == cudaSuccess) e = cudaMalloc(&nrows, sizeof(int) * (size_t)pcap);
    if (e == cudaSuccess) e = cudaMalloc(&nverts, sizeof(int) * (size_t)pcap);
  }
  if (e == cudaSuccess && vcap != scene->vcap) { verts = nullptr; e = cudaMalloc(&verts, sizeof(double) * vcap); }
  if (e == cudaSuccess && cap != scene->cap) { cols = nullptr; e = cudaMalloc(&cols, sizeof(double) * 6 * (size_t)cap); }
  if (e == cudaSuccess) {
    const double* vsrc = (const double*)(d + o_verts);
    const int* nvsrc = (const int*)(d + o_nverts);
    k_scene_ingest_polytopes<<<(cap + 7) / 8, 256, 0, st>>>(
        (const double*)d, (const int*)(d + o_nrows), vsrc, nvsrc, vin, total, vmax_new, cap, 0.0, rows, nrows, verts,
        nverts, cols, (const int*)(d + o_off), n_scenes, scene->seg_off);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);      // (the pinned staging is reused by the next update)
  // release whichever of each pair is not kept: the new buffers on failure, the replaced ones on success
  const bool ok = e == cudaSuccess;
  if (rows != scene->rows) {
    cudaFree(ok ? scene->rows : rows); cudaFree(ok ? scene->nrows : nrows); cudaFree(ok ? scene->nverts : nverts);
  }
  if (verts != scene->verts) cudaFree(ok ? scene->verts : verts);
  if (cols != scene->cols) cudaFree(ok ? scene->cols : cols);
  if (!ok) return bp_fail("bp_scene_update_polytopes_batch", e);
  scene->rows = rows; scene->nrows = nrows; scene->nverts = nverts; scene->pcap = pcap;
  scene->verts = verts; scene->vcap = vcap;
  scene->cols = cols; scene->cap = cap;
  scene->vmax = vmax_new;
  scene->n = n_max;
  memcpy(scene->seg_off_host, offsets_host, sizeof(int) * (size_t)(n_scenes + 1));
  return 0;
}

int bp_scene_destroy(bp_scene* scene) {
  if (!scene) return 0;
  if (scene->seg_off_host) free(scene->seg_off_host);
  if (scene->stage_h) cudaFreeHost(scene->stage_h);
  if (scene->stage_d) cudaFree(scene->stage_d);
  if (scene->seg_off) cudaFree(scene->seg_off);
  if (scene->rows) cudaFree(scene->rows);
  if (scene->nrows) cudaFree(scene->nrows);
  if (scene->verts) cudaFree(scene->verts);
  if (scene->nverts) cudaFree(scene->nverts);
  if (scene->cols) cudaFree(scene->cols);
  free(scene);
  return 0;
}

int bp_scene_size(const bp_scene* scene) { return scene ? scene->n : -1; }

int bp_closest_points(const bp_scene* scene, const double* seeds_dev, const double* q_inv_dev, int S,
                      double* y_out_dev, double* dist_out_dev, void* stream) {
  if (!scene || S < 0 || scene->seg_off) return bp_fail("bp_closest_points: bad arguments");
  if (S == 0 || scene->n == 0) return 0;
  dim3 grid((scene->n + 255) / 256, S);
  k_closest_points<<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(scene), seeds_dev, q_inv_dev, y_out_dev, dist_out_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_closest_points_line(const bp_scene* scene, const double* p0_dev, const double* p1_dev, int S,
                           double* x_out_dev, double* phi_out_dev, void* stream) {
  if (!scene || S < 0 || scene->seg_off) return bp_fail("bp_closest_points_line: bad arguments");
  if (S == 0 || scene->n == 0) return 0;
  dim3 grid((scene->n + 255) / 256, S);
  k_closest_points_line<<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(scene), p0_dev, p1_dev, x_out_dev, phi_out_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_polyhedron(const bp_scene* scene, const double* seeds_dev, const double* q_inv_dev, const double* q_ellipse_dev,
                  const double* init_rows_dev, int S, int m_max, double* A_dev, double* b_dev, int* m_dev,
                  int* status_dev, void* stream) {
  (void)q_inv_dev;   // the pass metric is derived from q_ellipse (= q_inv^-1, :227-228)
  if (!scene || S < 0 || m_max < 6 || m_max > BP_MAX_ROWS || scene->seg_off)
    return bp_fail("bp_polyhedron: bad arguments");
  if (S == 0) return 0;
  PolyParams pr;
  memset(&pr, 0, sizeof(pr));
  pr.seeds = seeds_dev; pr.q_ellipse = q_ellipse_dev; pr.init_rows = init_rows_dev;
  pr.A = A_dev; pr.b = b_dev; pr.m = m_dev; pr.status = status_dev; pr.m_max = m_max; pr.mode = 0;
  pr.cache_y = poly_cache_y(scene->n);
  pr.shell = !scene->rows && poly_point_shell(scene->n);
  size_t smem = poly_point_smem_bytes(scene->n, scene->rows != nullptr);
  if (scene->rows) {
    if (scene->n > BP_POLY_SCENE_MAX) return bp_fail("polytope scenes hold at most 16384 obstacles");
    if (set_dyn_smem((const void*)k_poly_point<true>, smem)) return 1;
    k_poly_point<true><<<S, poly_threads(scene->n), smem, (cudaStream_t)stream>>>(view_of(scene), pr);
  } else {
    if (set_dyn_smem((const void*)k_poly_point<false>, smem)) return 1;
    k_poly_point<false><<<S, poly_threads(scene->n), smem, (cudaStream_t)stream>>>(view_of(scene), pr);
  }
  BP_CUDA(cudaGetLastError());
  return 0;
}

static int launch_mvie(const MvieParams& pr, cudaStream_t stream) {
  k_mvie<<<pr.S, 32, 0, stream>>>(pr);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_mvie(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, int free_centre,
            const double* centre_dev, double* q_inv_out_dev, double* q_ellipse_out_dev, double* centre_out_dev,
            int* status_dev, int* newton_iters_dev, void* stream) {
  if (S < 0 || m_max < 1 || m_max > BP_MAX_ROWS) return bp_fail("bp_mvie: bad arguments");
  if (S == 0) return 0;
  MvieParams pr;
  memset(&pr, 0, sizeof(pr));
  pr.A = A_dev; pr.b = b_dev; pr.m = m_dev; pr.S = S; pr.m_max = m_max; pr.mode = 3; pr.free_centre = free_centre;
  pr.centre = centre_dev; pr.q_inv_out = q_inv_out_dev; pr.q_ellipse_out = q_ellipse_out_dev;
  pr.centre_out = centre_out_dev; pr.status_out = status_dev; pr.iters_out = newton_iters_dev;
  return launch_mvie(pr, (cudaStream_t)stream);
}

int bp_mvie_fixed_r(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max,
                    const double* centre_dev, const double* r_ellipse_dev, const double* a_lb_dev,
                    double* q_inv_out_dev, double* q_ellipse_out_dev, double* eigs_out_dev, int* status_dev,
                    int* newton_iters_dev, void* stream) {
  if (S < 0 || m_max < 1 || m_max > BP_MAX_ROWS) return bp_fail("bp_mvie_fixed_r: bad arguments");
  if (S == 0) return 0;
  k_mvie_fixed_r<<<S, 32, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, m_max, centre_dev, r_ellipse_dev, a_lb_dev,
                                                     q_inv_out_dev, q_ellipse_out_dev, eigs_out_dev, status_dev,
                                                     newton_iters_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_build_sets_around_line(const bp_scene* scene, const double* p0_dev, const double* dp1_dev, int S,
                              const double* ws_min_host, const double* ws_max_host, int optimize, int max_iter,
                              int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                              double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                              void* stream) {
  if (!scene || scene->seg_off || S < 0 || m_max < 6 || m_max > BP_MAX_ROWS || max_iter < 1 || !ws_min_host ||
      !ws_max_host)
    return bp_fail("bp_build_sets_around_line: bad arguments");
  if (S == 0) return 0;
  if (scene->n > 64 * 128) return bp_fail("bp_build_sets_around_line: scene too large (N > 8192)");
  FusedParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.seeds = p0_dev; fp.dp1 = dp1_dev;
  for (int i = 0; i < 3; ++i) { fp.ws_rows[2 * i] = ws_max_host[i]; fp.ws_rows[2 * i + 1] = -ws_min_host[i]; }
  fp.A = A_dev; fp.b = b_dev; fp.m = m_dev; fp.q_ellipse = q_ellipse_dev; fp.p_mid = p_mid_dev;
  fp.status = status_dev; fp.iters = iters_dev; fp.rows_peak = rows_peak_dev;
  fp.m_max = m_max; fp.max_iter = max_iter; fp.fixed_mid = 0; fp.optimize = optimize;
  fp.row_cap = row_cap; fp.cache_y = poly_cache_y(scene->n);
  const size_t fsmem = poly_smem_bytes(scene->n, scene->rows != nullptr);
  if (scene->rows) {
    if (scene->n > 64 * 128) return bp_fail("bp_build_sets_around_line: polytope scenes of at most 8192 obstacles");
    if (set_dyn_smem((const void*)k_iris_fused<1, true>, fsmem)) return 1;
    k_iris_fused<1, true><<<S, 128, fsmem, (cudaStream_t)stream>>>(view_of(scene), fp);
  } else {
    if (set_dyn_smem((const void*)k_iris_fused<1, false>, fsmem)) return 1;
    k_iris_fused<1, false><<<S, 128, fsmem, (cudaStream_t)stream>>>(view_of(scene), fp);
  }
  BP_CUDA(cudaGetLastError());
  return 0;
}

size_t bp_build_sets_workspace_bytes(int S) { return sizeof(SeedState) * (size_t)(S > 0 ? S : 1); }

int bp_build_sets_point(const bp_scene* scene, const double* seeds_dev, int S, const double* ws_min_host,
                        const double* ws_max_host, int fixed_mid, int optimize, int max_iter, int m_max,
                        double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev, double* p_mid_dev,
                        int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap, void* workspace_dev,
                        size_t workspace_bytes, void* stream_) {
  return bp_build_sets_point_ms(scene, nullptr, seeds_dev, S, ws_min_host, ws_max_host, fixed_mid, optimize, max_iter,
                                m_max, A_dev, b_dev, m_dev, q_ellipse_dev, p_mid_dev, status_dev, iters_dev,
                                rows_peak_dev, row_cap, workspace_dev, workspace_bytes, stream_);
}

int bp_build_sets_point_ms(const bp_scene* scene, const int* seed_scene_dev, const double* seeds_dev, int S,
                           const double* ws_min_host, const double* ws_max_host, int fixed_mid, int optimize,
                           int max_iter, int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                           double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                           void* workspace_dev, size_t workspace_bytes, void* stream_) {
  return bp_build_sets_point_x(scene, seed_scene_dev, seeds_dev, S, ws_min_host, ws_max_host, fixed_mid, optimize,
                               max_iter, m_max, A_dev, b_dev, m_dev, q_ellipse_dev, p_mid_dev, status_dev, iters_dev,
                               rows_peak_dev, row_cap, nullptr, nullptr, 0, 0, 0, 0, 0, 0, workspace_dev,
                               workspace_bytes, stream_);
}

int bp_build_sets_point_x(const bp_scene* scene, const int* seed_scene_dev, const double* seeds_dev, int S,
                          const double* ws_min_host, const double* ws_max_host, int fixed_mid, int optimize,
                          int max_iter, int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                          double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                          double* aabb_dev, const unsigned long long* peer_base_dev, int world, int slot0,
                          size_t off_A, size_t off_b, size_t off_m, size_t off_aabb, void* workspace_dev,
                          size_t workspace_bytes, void* stream_) {
  return bp_build_sets_point_tail(scene, seed_scene_dev, seeds_dev, S, ws_min_host, ws_max_host, fixed_mid, optimize,
                                  max_iter, m_max, A_dev, b_dev, m_dev, q_ellipse_dev, p_mid_dev, status_dev, iters_dev,
                                  rows_peak_dev, row_cap, aabb_dev, peer_base_dev, world, slot0, off_A, off_b, off_m,
                                  off_aabb, nullptr, workspace_dev, workspace_bytes, stream_);
}

int bp_step_begin(const bp_tail* tail, int double_buffered, void* stream_) {
  if (!tail || !tail->epoch || !tail->bits || tail->S_glob < 1 || tail->words < 1) return bp_fail("bp_step_begin: bad arguments");
  cudaStream_t stream = (cudaStream_t)stream_;
  const size_t n = (size_t)tail->S_glob * tail->words;
  int ctas = (int)((n + 255) / 256);
  if (ctas > 296) ctas = 296;
  k_step_begin<<<ctas, 256, 0, stream>>>(tail->epoch, tail->bits, n, double_buffered);
  k_step_epoch<<<1, 1, 0, stream>>>(tail->epoch);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_build_sets_point_tail(const bp_scene* scene, const int* seed_scene_dev, const double* seeds_dev, int S,
                             const double* ws_min_host, const double* ws_max_host, int fixed_mid, int optimize,
                             int max_iter, int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                             double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                             double* aabb_dev, const unsigned long long* peer_base_dev, int world, int slot0,
                             size_t off_A, size_t off_b, size_t off_m, size_t off_aabb, const bp_tail* tail,
                             void* workspace_dev, size_t workspace_bytes, void* stream_) {
  if (world < 0 || slot0 < 0 || (world > 0 && !peer_base_dev))
    return bp_fail("bp_build_sets_point_x: bad peer arguments");
  if (tail && (tail->S_glob < S || tail->S_glob > 128 * 64 || tail->words < (tail->S_glob + 31) / 32 || !tail->A ||
               !tail->b || !tail->m || !tail->aabb || !tail->count || !tail->log || !tail->bits || !tail->epoch ||
               !aabb_dev))
    return bp_fail("bp_build_sets_point_tail: bad tail arguments");
  if (scene && ((scene->seg_off != nullptr) != (seed_scene_dev != nullptr)))
    return bp_fail("bp_build_sets_point: a scene batch needs seed_scene, a single scene must not have it");
  if (!scene || S < 0 || m_max < 6 || m_max > BP_MAX_ROWS || max_iter < 1 || !ws_min_host || !ws_max_host)
    return bp_fail("bp_build_sets_point: bad arguments");
  if (S == 0) return 0;
  if (workspace_bytes < bp_build_sets_workspace_bytes(S)) return bp_fail("bp_build_sets_point: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  if (use_fused_iris(scene->n) && !(scene->rows && scene->n > 64 * 128)) {   // (polytope kernels: one word of alive bits)
    FusedParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.seeds = seeds_dev;
    for (int i = 0; i < 3; ++i) { fp.ws_rows[2 * i] = ws_max_host[i]; fp.ws_rows[2 * i + 1] = -ws_min_host[i]; }
    fp.A = A_dev; fp.b = b_dev; fp.m = m_dev; fp.q_ellipse = q_ellipse_dev; fp.p_mid = p_mid_dev;
    fp.status = status_dev; fp.iters = iters_dev; fp.rows_peak = rows_peak_dev;
    fp.m_max = m_max; fp.max_iter = max_iter; fp.fixed_mid = fixed_mid; fp.optimize = optimize;
    fp.row_cap = row_cap; fp.cache_y = poly_cache_y(scene->n);
    fp.aabb = aabb_dev;
    fp.peers.base = peer_base_dev; fp.peers.world = world; fp.peers.slot0 = slot0;
    fp.peers.off_A = off_A; fp.peers.off_b = off_b; fp.peers.off_m = off_m; fp.peers.off_aabb = off_aabb;
    if (tail) {
      fp.tail.S = tail->S_glob; fp.tail.words = tail->words;
      fp.tail.A = tail->A; fp.tail.b = tail->b; fp.tail.m = tail->m; fp.tail.aabb = tail->aabb;
      fp.tail.count = tail->count; fp.tail.log = tail->log; fp.tail.bits = tail->bits; fp.tail.epoch = tail->epoch;
      fp.tail.off_count = tail->off_count; fp.tail.off_log = tail->off_log; fp.tail.off_bits = tail->off_bits;
      fp.tail.tol = tail->tol;
    }
    size_t fsmem = poly_smem_bytes(scene->n, scene->rows != nullptr);
    // box scenes small enough for two CTAs per SM: the scene columns are staged in shared memory by TMA
    // (BPGEO_STAGE=0 keeps the global / L1 loads: the A/B switch of profiles/r02_stage_ab.txt)
    {
      static int env = -1;
      if (env < 0) { const char* e = getenv("BPGEO_STAGE"); env = (e && e[0] == '0') ? 0 : 1; }
      const size_t staged = 16 * ((sizeof(ShellMem) + 15) / 16) + sizeof(double) * (size_t)((scene->n + 1) & ~1) * 7;
      if (env && !scene->rows && staged + 20 * 1024 <= 110 * 1024) { fp.stage = 1; fsmem = staged; }
    }
    // (speculative trailing solve: decided below, box scenes only)
    const void* kfn = scene->rows ? (const void*)k_iris_fused<0, true>
                      : (scene->n <= 64 * 128 ? (const void*)k_iris_fused<0, false>
                                              : (const void*)k_iris_fused<0, false, 2>);   // (2 words of alive bits)
    if (tail && fsmem < sizeof(double) * BP_TAIL_WORK_DOUBLES) fsmem = sizeof(double) * BP_TAIL_WORK_DOUBLES;
    if (set_dyn_smem(kfn, fsmem)) return 1;
    {
      // speculative trailing solve on every pass: pays when the launch runs in waves (a seed that ends early hands
      // its slot to the next one sooner) AND the polyhedron passes carry the seed's time: the two solver warps of a
      // CTA slow each other down by ~15 % even on different sub-partitions.  Measured: C4 (10 k obstacles, 2048
      // seeds) 2.24 -> 2.09 ms, the C2 scene with 2048 seeds 1.82 -> 1.98 ms, C2 itself 0.43 -> 0.46 ms.  Hence on
      // for multi-wave launches over large scenes only; BPGEO_SPEC=0 / 1 forces it off / on.
      static int env = -2, resident = 0;
      if (env == -2) {
        const char* e = getenv("BPGEO_SPEC");
        env = e ? (e[0] == '0' ? 0 : 1) : -1;
        int dev = 0, nsm = 148;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
        resident = 2 * nsm;
      }
      fp.spec = env >= 0 ? env : ((S > resident && scene->n >= 4096) ? 1 : 0);
      if (scene->rows || tail) fp.spec = 0;
      if (fp.spec) {
        kfn = scene->n <= 64 * 128 ? (const void*)k_iris_fused<0, false, 1, true> : (const void*)k_iris_fused<0, false, 2, true>;
        if (set_dyn_smem(kfn, fsmem)) return 1;
      }
    }
    if (tail) {
      // the pair workers of the tail wait inside the kernel for the other sets: every CTA has to be resident
      int nb = 0, dev = 0, nsm = 0;
      BP_CUDA(cudaGetDevice(&dev));
      BP_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
      BP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, 128, fsmem));
      if ((long long)S > (long long)nb * nsm) {
        snprintf(g_err, sizeof(g_err), "bp_build_sets_point_tail: %d seeds exceed the %d CTAs that are resident at once", S,
                 nb * nsm);
        return 1;
      }
    }
    if (scene->rows) k_iris_fused<0, true><<<S, 128, fsmem, stream>>>(view_of(scene, seed_scene_dev), fp);
    else if (fp.spec && scene->n <= 64 * 128) k_iris_fused<0, false, 1, true><<<S, 128, fsmem, stream>>>(view_of(scene, seed_scene_dev), fp);
    else if (fp.spec) k_iris_fused<0, false, 2, true><<<S, 128, fsmem, stream>>>(view_of(scene, seed_scene_dev), fp);
    else if (scene->n <= 64 * 128) k_iris_fused<0, false><<<S, 128, fsmem, stream>>>(view_of(scene, seed_scene_dev), fp);
    else k_iris_fused<0, false, 2><<<S, 128, fsmem, stream>>>(view_of(scene, seed_scene_dev), fp);
    BP_CUDA(cudaGetLastError());
    return 0;
  }
  if (tail) return bp_fail("bp_build_sets_point_tail: the launch-sequence path (N > 16384 or BPGEO_FUSED=0) has no tail");
  SeedState* st = (SeedState*)workspace_dev;
  k_state_init<<<(S + 127) / 128, 128, 0, stream>>>(st, seeds_dev, S);
  PolyParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.state = st; pp.A = A_dev; pp.b = b_dev; pp.m = m_dev; pp.status = status_dev; pp.m_max = m_max;
  pp.mode = 1; pp.max_iter = max_iter;
  pp.row_cap = optimize ? row_cap : 0;
  for (int i = 0; i < 3; ++i) { pp.ws_rows[2 * i] = ws_max_host[i]; pp.ws_rows[2 * i + 1] = -ws_min_host[i]; }
  MvieParams mp;
  memset(&mp, 0, sizeof(mp));
  mp.A = A_dev; mp.b = b_dev; mp.m = m_dev; mp.S = S; mp.m_max = m_max; mp.state = st;
  pp.cache_y = poly_cache_y(scene->n);
  pp.shell = !scene->rows && poly_point_shell(scene->n);
  size_t smem = poly_point_smem_bytes(scene->n, scene->rows != nullptr);
  if (scene->rows && scene->n > BP_POLY_SCENE_MAX) return bp_fail("polytope scenes hold at most 16384 obstacles");
  if (set_dyn_smem(scene->rows ? (const void*)k_poly_point<true> : (const void*)k_poly_point<false>, smem)) return 1;
  const int T = poly_threads(scene->n);
  const int passes = optimize ? max_iter : 1;
  for (int it = 0; it < passes; ++it) {
    if (scene->rows) k_poly_point<true><<<S, T, smem, stream>>>(view_of(scene, seed_scene_dev), pp);
    else k_poly_point<false><<<S, T, smem, stream>>>(view_of(scene, seed_scene_dev), pp);
    if (!optimize) break;                                 // :214-215
    mp.mode = fixed_mid ? 0 : 1;
    if (launch_mvie(mp, stream)) return 1;
  }
  if (optimize && fixed_mid) {                            // :235-238
    mp.mode = 2;
    if (launch_mvie(mp, stream)) return 1;
  }
  k_state_export<<<(S + 127) / 128, 128, 0, stream>>>(st, S, optimize ? max_iter : 1 << 30, q_ellipse_dev, p_mid_dev, status_dev, iters_dev,
                                                      rows_peak_dev);
  // the launch-sequence path delivers boxes / peer copies with the stand-alone kernels
  if (world > 0 && !aabb_dev) return bp_fail("bp_build_sets_point_x: the launch-sequence path needs aabb_dev for the peer stores");
  if (aabb_dev) k_set_aabb<<<S, 128, 0, stream>>>(A_dev, b_dev, m_dev, S, m_max, aabb_dev);
  if (world > 0)
    k_scatter_sets_peers<<<S, 128, 0, stream>>>(A_dev, b_dev, m_dev, aabb_dev, m_max, slot0, peer_base_dev, world, off_A,
                                                off_b, off_m, off_aabb);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_build_sets_line(const bp_scene* scene, const double* p0_dev, const double* p1_dev, int S,
                       const double* ws_min_host, const double* ws_max_host, int limit_space, double e_max,
                       int compute_ellipsoid, int m_max, double* A_dev, double* b_dev, int* m_dev,
                       double* q_ellipse_dev, double* p_mid_dev, int* collision_dev, int* status_dev,
                       void* workspace_dev, size_t workspace_bytes, void* stream_) {
  return bp_build_sets_line_ms(scene, nullptr, p0_dev, p1_dev, S, ws_min_host, ws_max_host, limit_space, e_max,
                               compute_ellipsoid, m_max, A_dev, b_dev, m_dev, q_ellipse_dev, p_mid_dev, collision_dev,
                               status_dev, workspace_dev, workspace_bytes, stream_);
}

int bp_build_sets_line_ms(const bp_scene* scene, const int* seg_scene_dev, const double* p0_dev, const double* p1_dev,
                          int S, const double* ws_min_host, const double* ws_max_host, int limit_space, double e_max,
                          int compute_ellipsoid, int m_max, double* A_dev, double* b_dev, int* m_dev,
                          double* q_ellipse_dev, double* p_mid_dev, int* collision_dev, int* status_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream_) {
  if (scene && ((scene->seg_off != nullptr) != (seg_scene_dev != nullptr)))
    return bp_fail("bp_build_sets_line: a scene batch needs seg_scene, a single scene must not have it");
  if (!scene || S < 0 || m_max < 6 || m_max > BP_MAX_ROWS || !ws_min_host || !ws_max_host)
    return bp_fail("bp_build_sets_line: bad arguments");
  if (S == 0) return 0;
  if (compute_ellipsoid && workspace_bytes < bp_build_sets_workspace_bytes(S))
    return bp_fail("bp_build_sets_line: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  LineParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.p0 = p0_dev; lp.p1 = p1_dev; lp.limit_space = limit_space; lp.e_max = e_max;
  for (int i = 0; i < 3; ++i) { lp.ws_rows[2 * i] = ws_max_host[i]; lp.ws_rows[2 * i + 1] = -ws_min_host[i]; }
  lp.A = A_dev; lp.b = b_dev; lp.m = m_dev; lp.status = status_dev; lp.collision = collision_dev; lp.m_max = m_max;
  if (scene->rows) {                                     // general polytopes: dist | x[3] | p_closest[3] per obstacle
    lp.cache_x = scene->n <= 3072;
    const size_t psmem = sizeof(double) * (lp.cache_x ? 7 : 1) * (size_t)scene->n;
    if (scene->n > BP_POLY_SCENE_MAX) return bp_fail("polytope scenes hold at most 16384 obstacles");
    if (set_dyn_smem((const void*)k_poly_line_p, psmem)) return 1;
    k_poly_line_p<<<S, poly_threads(scene->n), psmem, stream>>>(view_of(scene, seg_scene_dev), lp);
  } else {
    size_t smem = sizeof(double) * (size_t)(scene->n > 0 ? scene->n : 1);
    if (set_dyn_smem((const void*)k_poly_line, smem)) return 1;
    k_poly_line<<<S, poly_threads(scene->n), smem, stream>>>(view_of(scene, seg_scene_dev), lp);
  }
  if (compute_ellipsoid) {
    SeedState* st = (SeedState*)workspace_dev;
    k_state_init_line<<<(S + 127) / 128, 128, 0, stream>>>(st, p0_dev, status_dev, S);
    MvieParams mp;
    memset(&mp, 0, sizeof(mp));
    mp.A = A_dev; mp.b = b_dev; mp.m = m_dev; mp.S = S; mp.m_max = m_max; mp.state = st; mp.mode = 2;
    if (launch_mvie(mp, stream)) return 1;
    k_state_export<<<(S + 127) / 128, 128, 0, stream>>>(st, S, 0, q_ellipse_dev, p_mid_dev, status_dev, nullptr, nullptr);
  }
  BP_CUDA(cudaGetLastError());
  return 0;
}

size_t bp_pair_workspace_bytes(int S, int rows) {
  if (S < 0) S = 0;
  if (rows < 0) rows = 0;
  // aabb [S,6] doubles | counter (16 B) | pair list: at most rows * S entries of int2
  return sizeof(double) * 6 * (size_t)S + 16 + sizeof(int2) * (size_t)rows * (size_t)S;
}

int bp_set_aabb(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double* aabb_out_dev,
                void* stream) {
  if (S < 0 || m_max < 1 || m_max > BP_MAX_ROWS || !aabb_out_dev) return bp_fail("bp_set_aabb: bad arguments");
  if (S == 0) return 0;
  k_set_aabb<<<S, 128, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, S, m_max, aabb_out_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

static int pair_feasible_impl(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double tol,
                              int row_begin, int row_end, unsigned int* adj_bits_dev, double* x_feas_dev,
                              const double* aabb_in_dev, void* workspace_dev, size_t workspace_bytes, void* stream_,
                              cudaEvent_t* ev) {
  if (S < 0 || row_begin < 0 || row_end > S || row_begin > row_end || m_max < 1 || m_max > BP_MAX_ROWS)
    return bp_fail("bp_pair_feasible: bad arguments");
  if (row_end == row_begin) return 0;
  const int rows = row_end - row_begin;
  if (workspace_bytes < bp_pair_workspace_bytes(S, rows)) return bp_fail("bp_pair_feasible: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  double* aabb = (double*)workspace_dev;
  unsigned int* count = (unsigned int*)(aabb + 6 * (size_t)S);
  int2* list = (int2*)((char*)count + 16);
  const int words = (S + 31) / 32;
  BP_CUDA(cudaMemsetAsync(adj_bits_dev, 0, sizeof(unsigned int) * (size_t)rows * words, stream));
  BP_CUDA(cudaMemsetAsync(count, 0, 16, stream));
  if (ev) BP_CUDA(cudaEventRecord(ev[0], stream));
  if (aabb_in_dev) aabb = const_cast<double*>(aabb_in_dev);      // boxes computed elsewhere (e.g. all-gathered)
  else k_set_aabb<<<S, 128, 0, stream>>>(A_dev, b_dev, m_dev, S, m_max, aabb);
  if (ev) BP_CUDA(cudaEventRecord(ev[1], stream));
  dim3 grid((S + 31) / 32, (rows + 7) / 8);
  k_pair_filter<<<grid, 256, 0, stream>>>(aabb, S, row_begin, row_end, list, count);
  if (ev) BP_CUDA(cudaEventRecord(ev[2], stream));
  int nsm = 148;
  {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  }
  const long long max_pairs = (long long)rows * S;
  long long ctas = (max_pairs + 7) / 8;              // 8 warps per CTA, one pair per warp per trip
  static int lp_ctas_per_sm = 0;                     // resident CTAs per SM (registers / shared memory)
  if (lp_ctas_per_sm == 0) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_pair_lp, 256, 0) != cudaSuccess || nb < 1) nb = 1;
    lp_ctas_per_sm = nb;
  }
  if (ctas > (long long)nsm * lp_ctas_per_sm) ctas = (long long)nsm * lp_ctas_per_sm;
  if (ctas < 1) ctas = 1;
  k_pair_lp<<<(int)ctas, 256, 0, stream>>>(A_dev, b_dev, m_dev, S, m_max, tol, row_begin, aabb, list, count, adj_bits_dev,
                                           x_feas_dev);
  if (ev) BP_CUDA(cudaEventRecord(ev[3], stream));
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_pair_feasible(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double tol,
                     int row_begin, int row_end, unsigned int* adj_bits_dev, double* x_feas_dev,
                     const double* aabb_in_dev, void* workspace_dev, size_t workspace_bytes, void* stream_) {
  return pair_feasible_impl(A_dev, b_dev, m_dev, S, m_max, tol, row_begin, row_end, adj_bits_dev, x_feas_dev, aabb_in_dev,
                            workspace_dev, workspace_bytes, stream_, nullptr);
}

int bp_pair_feasible_stages(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double tol,
                            int row_begin, int row_end, unsigned int* adj_bits_dev, const double* aabb_in_dev,
                            void* workspace_dev, size_t workspace_bytes, void* stream_, float* ms_host) {
  if (!ms_host) return bp_fail("bp_pair_feasible_stages: bad arguments");
  ms_host[0] = ms_host[1] = ms_host[2] = 0.f;
  if (row_end <= row_begin) return 0;
  cudaEvent_t ev[4];
  for (int k = 0; k < 4; ++k) BP_CUDA(cudaEventCreate(&ev[k]));
  int rc = pair_feasible_impl(A_dev, b_dev, m_dev, S, m_max, tol, row_begin, row_end, adj_bits_dev, nullptr, aabb_in_dev,
                              workspace_dev, workspace_bytes, stream_, ev);
  if (rc == 0) {
    BP_CUDA(cudaEventSynchronize(ev[3]));
    for (int k = 0; k < 3; ++k) BP_CUDA(cudaEventElapsedTime(&ms_host[k], ev[k], ev[k + 1]));
  }
  for (int k = 0; k < 4; ++k) cudaEventDestroy(ev[k]);
  return rc;
}

int bp_pairs_feasible_list(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double tol,
                           const int* pairs_dev, int P, int* result_dev, double* x_feas_dev, void* workspace_dev,
                           size_t workspace_bytes, void* stream_) {
  if (S < 0 || P < 0 || m_max < 1 || m_max > BP_MAX_ROWS || !result_dev) return bp_fail("bp_pairs_feasible_list: bad arguments");
  if (P == 0 || S == 0) return 0;
  if (workspace_bytes < sizeof(double) * 6 * (size_t)S) return bp_fail("bp_pairs_feasible_list: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  double* aabb = (double*)workspace_dev;
  k_set_aabb<<<S, 128, 0, stream>>>(A_dev, b_dev, m_dev, S, m_max, aabb);
  k_pair_list<<<(P + 7) / 8, 256, 0, stream>>>(A_dev, b_dev, m_dev, m_max, tol, aabb, (const int2*)pairs_dev, P,
                                               result_dev, x_feas_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

size_t bp_sets_obstacles_workspace_bytes(int S) { return sizeof(double) * 6 * (size_t)(S > 0 ? S : 0); }

int bp_sets_obstacles(const bp_scene* scene, const int* set_scene_dev, const double* A_dev, const double* b_dev,
                      const int* m_dev, int S, int m_max, double tol, int* first_hit_dev, void* workspace_dev,
                      size_t workspace_bytes, void* stream_) {
  if (!scene || S < 0 || m_max < 1 || m_max > BP_MAX_ROWS) return bp_fail("bp_sets_obstacles: bad arguments (m_max 1 .. 48)");
  if (!(tol >= 0.0) || !isfinite(tol)) return bp_fail("bp_sets_obstacles: tol must be finite and >= 0");
  if (S == 0) return 0;
  if (!A_dev || !b_dev || !m_dev || !first_hit_dev) return bp_fail("bp_sets_obstacles: bad arguments");
  if (!workspace_dev || workspace_bytes < bp_sets_obstacles_workspace_bytes(S))
    return bp_fail("bp_sets_obstacles: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  double* aabb = (double*)workspace_dev;
  k_set_aabb<<<S, 128, 0, stream>>>(A_dev, b_dev, m_dev, S, m_max, aabb);
  k_sets_obstacles<<<(S + 7) / 8, 256, 0, stream>>>(view_of(scene), scene->seg_off ? scene->n_seg : 1, set_scene_dev,
                                                    A_dev, b_dev, m_dev, S, m_max, tol, aabb, first_hit_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_reduce_ineqs(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double* A_out_dev,
                    double* b_out_dev, int* m_out_dev, unsigned char* keep_out_dev, int* status_dev, void* stream) {
  if (S == 0) return 0;                       // an empty batch has no buffers
  if (S < 0 || m_max < 1 || m_max > BP_MAX_ROWS || !A_out_dev || !b_out_dev || !m_out_dev)
    return bp_fail("bp_reduce_ineqs: bad arguments");
  k_reduce_rows<<<S, 128, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, m_max, A_out_dev, b_out_dev, m_out_dev,
                                                      keep_out_dev, status_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_polytope_vertices(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, int vmax,
                         double* V_dev, int* nv_dev, int* status_dev, void* stream) {
  if (S < 0 || m_max < 1 || m_max > BP_MAX_ROWS || vmax < 1 || !V_dev || !nv_dev || !status_dev)
    return bp_fail("bp_polytope_vertices: bad arguments");
  if (S == 0) return 0;
  k_polytope_vertices<<<S, 128, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, m_max, vmax, V_dev, nv_dev, status_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_check_fit(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, const int* pairs_dev,
                 int P, const double* x0_dev, const int* active_dev, const double* l_ee_samples_host, int n_samples,
                 double margin, int* fits_dev, int* first_sample_dev, void* stream) {
  if (S < 0 || P < 0 || m_max < 1 || m_max > BP_MAX_ROWS || n_samples < 1 || n_samples > BP_FIT_SAMPLES ||
      !l_ee_samples_host || !fits_dev || !first_sample_dev)
    return bp_fail("bp_check_fit: bad arguments");
  if (P == 0) return 0;
  FitParams fp;
  memset(&fp, 0, sizeof(fp));
  for (int k = 0; k < n_samples; ++k)
    for (int c = 0; c < 3; ++c) fp.l[k][c] = l_ee_samples_host[3 * k + c];
  fp.margin = margin;
  fp.n_samples = n_samples;
  for (int k = 0; k < n_samples; ++k) {           // distinct offsets (bitwise), first occurrence each
    bool seen = false;
    for (int q = 0; q < fp.nu && !seen; ++q)
      seen = memcmp(fp.l[fp.uidx[q]], fp.l[k], sizeof(double) * 3) == 0;
    if (!seen) fp.uidx[fp.nu++] = k;
  }
  BP_CUDA(cudaMemsetAsync(first_sample_dev, 0x7f, sizeof(int) * (size_t)P, (cudaStream_t)stream));
  const long long warps = (long long)P * fp.nu;
  k_fit_check<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, m_max,
                                                                             (const int2*)pairs_dev, P, x0_dev, active_dev,
                                                                             fp, first_sample_dev);
  k_fit_finish<<<(P + 127) / 128, 128, 0, (cudaStream_t)stream>>>(m_dev, (const int2*)pairs_dev, P, active_dev, n_samples,
                                                                   fits_dev, first_sample_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_project_points(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max,
                      const int* pairs_dev, int P, const double* xd_dev, double* x_out_dev, int* status_dev,
                      void* stream) {
  if (S < 0 || P < 0 || m_max < 1 || m_max > BP_MAX_ROWS || !xd_dev || !x_out_dev)
    return bp_fail("bp_project_points: bad arguments");
  if (P == 0) return 0;
  k_project<<<(P + 7) / 8, 256, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, m_max, (const int2*)pairs_dev, P,
                                                           xd_dev, x_out_dev, status_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_sample_filter(const bp_scene* scene, const int* item_scene_dev, const double* cand_dev, int Q, int C,
                     const double* A_dev, const double* b_dev, const int* m_dev, int m_max, const int* set_off_dev,
                     int* first_ok_dev, unsigned char* flags_dev, void* stream) {
  if (!scene || Q < 0 || C < 1 || !cand_dev || !first_ok_dev || (set_off_dev && (m_max < 1 || !A_dev || !b_dev || !m_dev)))
    return bp_fail("bp_sample_filter: bad arguments");
  if ((scene->seg_off != nullptr) != (item_scene_dev != nullptr))
    return bp_fail("bp_sample_filter: a scene batch needs item_scene, a single scene must not have it");
  if (Q == 0) return 0;
  k_sample_filter<<<Q, 128, 0, (cudaStream_t)stream>>>(view_of(scene, item_scene_dev), cand_dev, C, A_dev, b_dev, m_dev,
                                                       m_max, set_off_dev, nullptr, first_ok_dev, flags_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_sample_filter_tables(const bp_scene* scene, const int* item_scene_dev, const double* cand_dev, int Q, int C,
                            const double* A_dev, const double* b_dev, const int* m_dev, int m_max,
                            const int* set_begin_dev, const int* set_count_dev, int* first_ok_dev, void* stream) {
  if (!scene || Q < 0 || C < 1 || !cand_dev || !first_ok_dev || m_max < 1 || !A_dev || !b_dev || !m_dev ||
      !set_begin_dev || !set_count_dev)
    return bp_fail("bp_sample_filter_tables: bad arguments");
  if ((scene->seg_off != nullptr) != (item_scene_dev != nullptr))
    return bp_fail("bp_sample_filter_tables: a scene batch needs item_scene, a single scene must not have it");
  if (Q == 0) return 0;
  k_sample_filter<<<Q, 128, 0, (cudaStream_t)stream>>>(view_of(scene, item_scene_dev), cand_dev, C, A_dev, b_dev, m_dev,
                                                       m_max, set_begin_dev, set_count_dev, first_ok_dev, nullptr);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_dedupe_distance(const double* q_new_dev, const double* p_new_dev, int P, const double* q_nodes_dev,
                       const double* p_nodes_dev, const int* node_off_dev, double* dmin_dev, int* argmin_dev,
                       void* stream) {
  if (P < 0 || !q_new_dev || !p_new_dev || !node_off_dev || !dmin_dev) return bp_fail("bp_dedupe_distance: bad arguments");
  if (P == 0) return 0;
  k_dedupe_dist<<<P, 32, 0, (cudaStream_t)stream>>>(q_new_dev, p_new_dev, q_nodes_dev, p_nodes_dev, node_off_dev,
                                                    nullptr, dmin_dev, argmin_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_dedupe_distance_tables(const double* q_new_dev, const double* p_new_dev, int P, const double* q_nodes_dev,
                              const double* p_nodes_dev, const int* node_begin_dev, const int* node_count_dev,
                              double* dmin_dev, int* argmin_dev, void* stream) {
  if (P < 0 || !q_new_dev || !p_new_dev || !node_begin_dev || !node_count_dev || !dmin_dev)
    return bp_fail("bp_dedupe_distance_tables: bad arguments");
  if (P == 0) return 0;
  k_dedupe_dist<<<P, 32, 0, (cudaStream_t)stream>>>(q_new_dev, p_new_dev, q_nodes_dev, p_nodes_dev, node_begin_dev,
                                                    node_count_dev, dmin_dev, argmin_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_shortest_paths(const int* node_off_dev, const int* edge_off_dev, const int* edge_dst_dev,
                      const double* edge_w_dev, const int* src_dev, const int* dst_dev, int G, int max_len,
                      int* path_dev, int* path_len_dev, double* cost_dev, void* stream) {
  if (G < 0 || max_len < 1 || !node_off_dev || !edge_off_dev || !src_dev || !dst_dev || !path_dev || !path_len_dev ||
      !cost_dev)
    return bp_fail("bp_shortest_paths: bad arguments");
  if (G == 0) return 0;
  k_shortest_path<<<G, 32, 0, (cudaStream_t)stream>>>(node_off_dev, edge_off_dev, edge_dst_dev, edge_w_dev, src_dev,
                                                      dst_dev, max_len, path_dev, path_len_dev, cost_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_scatter_sets_peers(const double* A_dev, const double* b_dev, const int* m_dev, const double* aabb_dev, int S_loc,
                          int m_max, int slot0, const unsigned long long* peer_base_dev, int world, size_t off_A,
                          size_t off_b, size_t off_m, size_t off_aabb, void* stream) {
  if (S_loc < 0 || m_max < 1 || m_max > BP_MAX_ROWS || slot0 < 0 || world < 1 || !peer_base_dev || !A_dev || !b_dev ||
      !m_dev || !aabb_dev)
    return bp_fail("bp_scatter_sets_peers: bad arguments");
  if (S_loc == 0) return 0;
  k_scatter_sets_peers<<<S_loc, 128, 0, (cudaStream_t)stream>>>(A_dev, b_dev, m_dev, aabb_dev, m_max, slot0, peer_base_dev,
                                                                world, off_A, off_b, off_m, off_aabb);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_scatter_rows_peers(const unsigned int* rows_dev, int rows, int words, int row0,
                          const unsigned long long* peer_base_dev, int world, size_t off_bits, void* stream) {
  if (rows < 0 || words < 1 || row0 < 0 || world < 1 || !peer_base_dev) return bp_fail("bp_scatter_rows_peers: bad arguments");
  if (rows == 0) return 0;
  const size_t n = (size_t)rows * words;
  int ctas = (int)((n + 255) / 256);
  if (ctas > 1184) ctas = 1184;
  k_scatter_rows_peers<<<ctas, 256, 0, (cudaStream_t)stream>>>(rows_dev, rows, words, row0, peer_base_dev, world, off_bits);
  BP_CUDA(cudaGetLastError());
  return 0;
}

int bp_fk_iiwa14(const double* q_dev, int B, double* p_ee_dev, double* p_col_dev, double* T_ee_dev, double* jac_dev,
                 void* stream) {
  if (B < 0 || !p_ee_dev || !p_col_dev) return bp_fail("bp_fk_iiwa14: bad arguments");
  if (B == 0) return 0;
  // bulk (TMA) copies need 16-byte aligned global addresses; every tile offset is a multiple of 16 bytes
  const uintptr_t al = (uintptr_t)q_dev | (uintptr_t)p_ee_dev | (uintptr_t)p_col_dev | (uintptr_t)T_ee_dev |
                       (uintptr_t)jac_dev;
  const int use_tma = (al & 15) == 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (T_ee_dev && jac_dev) return launch_fk<true, true>(q_dev, B, p_ee_dev, p_col_dev, T_ee_dev, jac_dev, use_tma, st);
  if (T_ee_dev) return launch_fk<true, false>(q_dev, B, p_ee_dev, p_col_dev, T_ee_dev, jac_dev, use_tma, st);
  if (jac_dev) return launch_fk<false, true>(q_dev, B, p_ee_dev, p_col_dev, T_ee_dev, jac_dev, use_tma, st);
  return launch_fk<false, false>(q_dev, B, p_ee_dev, p_col_dev, T_ee_dev, jac_dev, use_tma, st);
}

int bp_debug_counters(unsigned long long* out_host, int n, int reset) {
  if (!out_host || n < 1) return bp_fail("bp_debug_counters: bad arguments");
  unsigned long long v = 0ull;
  BP_CUDA(cudaMemcpyFromSymbol(&v, g_shell_fallbacks, sizeof(v)));
  out_host[0] = v;
  for (int k = 1; k < n; ++k) out_host[k] = 0ull;
  if (reset) {
    v = 0ull;
    BP_CUDA(cudaMemcpyToSymbol(g_shell_fallbacks, &v, sizeof(v)));
  }
  return 0;
}

int bp_fk_iiwa14_kin(const double* q_dev, const double* dq_dev, int B, double* T_ee_dev, double* jac_dev,
                     double* djac_dev, void* stream) {
  if (B < 0 || !q_dev || !T_ee_dev || !jac_dev || (djac_dev && !dq_dev)) return bp_fail("bp_fk_iiwa14_kin: bad arguments");
  if (B == 0) return 0;
  k_fk_kin<<<(B + 31) / 32, 32, 0, (cudaStream_t)stream>>>(q_dev, dq_dev, B, T_ee_dev, jac_dev, djac_dev);
  BP_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"

// Native lock-step planner driver (bp_plan_create / bp_plan_run / bp_plan_destroy).
#include "bp_plan_gpu.cuh"

// ---------------------------------------------------------------------------
// Diagnostics: FP64 pipe probe used by bench.py for the roofline denominator.
// chains independent DFMA chains per thread, iters steps each.
// ---------------------------------------------------------------------------
template <int CHAINS>
__global__ void k_probe_fp64(double* out, int iters, double a, double b) {
  double x[CHAINS];
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) x[c] = 1.0 + 1e-3 * (threadIdx.x + c);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int c = 0; c < CHAINS; ++c) x[c] = fma(x[c], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) s += x[c];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" int bp_probe_fp64(int chains, int blocks, int threads, int iters, double* out_dev, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (chains == 1) k_probe_fp64<1><<<blocks, threads, 0, st>>>(out_dev, iters, 0.999999, 1e-9);
  else if (chains == 4) k_probe_fp64<4><<<blocks, threads, 0, st>>>(out_dev, iters, 0.999999, 1e-9);
  else if (chains == 8) k_probe_fp64<8><<<blocks, threads, 0, st>>>(out_dev, iters, 0.999999, 1e-9);
  else return bp_fail("bp_probe_fp64: chains must be 1, 4 or 8");
  BP_CUDA(cudaGetLastError());
  return 0;
}
