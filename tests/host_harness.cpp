// tests/host_harness.cpp -- TEST-ONLY host build of the thread-serial device
// primitives (csrc/bp_*.cuh are __host__ __device__).  It lets the CPU test
// suite check the exact code that runs inside the kernels against the oracle
// without a GPU.  It is NOT part of the product: boundplanner_b200/ never
// loads it and libbpgeo.so has no CPU path.
#include "../boundplanner_b200/csrc/bp_math.cuh"
#include "../boundplanner_b200/csrc/bp_mvie.cuh"
#include "../boundplanner_b200/csrc/bp_mvie_fixed_r.cuh"
#include "../boundplanner_b200/csrc/bp_mvie_pd.cuh"
#include "../boundplanner_b200/csrc/bp_lp.cuh"
#include "../boundplanner_b200/csrc/bp_fk.cuh"
#include "../boundplanner_b200/csrc/bp_planner.h"

struct HostRows {
  const double* A;   // [m,3]
  const double* B;   // [m]
  double a(int i, int k) const { return A[3 * i + k]; }
  double b(int i) const { return B[i]; }
};

extern "C" {

int hh_mvie(const double* A, const double* b, int m, int free_centre, const double* c0, double* E, double* Q,
            double* centre, int* iters) {
  HostRows rows{A, b};
  double L[6], d[3];
  int st = free_centre ? bp_mvie_solve<9>(rows, m, c0, L, d, iters) : bp_mvie_solve<6>(rows, m, c0, L, d, iters);
  double det;
  bp_shape_from_L(L, E, Q, &det);
  centre[0] = d[0]; centre[1] = d[1]; centre[2] = d[2];
  return st;
}

int hh_mvie_ws(const double* A, const double* b, int m, int free_centre, const double* c0, const double* L0, double t0,
               double* E, double* Lout, double* centre, int* iters) {
  HostRows rows{A, b};
  double L[6], d[3];
  int st = free_centre ? bp_mvie_solve<9>(rows, m, c0, L, d, iters, L0, t0)
                       : bp_mvie_solve<6>(rows, m, c0, L, d, iters, L0, t0);
  double Q[9], det;
  bp_shape_from_L(L, E, Q, &det);
  for (int k = 0; k < 6; ++k) Lout[k] = L[k];
  centre[0] = d[0]; centre[1] = d[1]; centre[2] = d[2];
  return st;
}

// hybrid barrier / primal-dual MVIE (bp_mvie_pd.cuh, the specification of the next solver); phase_iters[3] =
// Newton iterations of the barrier centring, the primal-dual phase and the final barrier stages
int hh_mvie_pd(const double* A, const double* b, int m, int free_centre, const double* c0, double* E, double* Q,
               double* centre, int* iters, int* phase_iters) {
  HostRows rows{A, b};
  double L[6], d[3];
  BpQ4 z[48];                                  // BP_MAX_ROWS of include/bpgeo.h
  if (m > 48) return BP_ROW_OVERFLOW;
  int st = free_centre ? bp_mvie_pd_solve<9>(rows, m, c0, L, d, iters, z, phase_iters)
                       : bp_mvie_pd_solve<6>(rows, m, c0, L, d, iters, z, phase_iters);
  double det;
  bp_shape_from_L(L, E, Q, &det);
  centre[0] = d[0]; centre[1] = d[1]; centre[2] = d[2];
  return st;
}

// fixed-rotation MVIE (mvie_socp_fixed_r): E = q_new, Q = q_ellipse, eigs = semi-axes
int hh_mvie_fixed_r(const double* A, const double* b, int m, const double* p_mid, const double* R, double a_lb,
                    double* E, double* Q, double* eigs, int* iters) {
  HostRows rows{A, b};
  BpSerialRed red;
  int st = bp_mvie_fixed_r(rows, m, p_mid, R, a_lb, red, eigs, iters);
  if (st == BP_OK) bp_shape_from_axes(R, eigs, E, Q, nullptr);
  return st;
}

void hh_line_frame(const double* dp1, double* R, double* l_seg) { bp_line_frame(dp1, R, l_seg); }

// closest points of n boxes to p in the metric of E (q_inv): y[n,3], dist[n]
void hh_box_qp(const double* E, const double* p, const double* lb, const double* ub, int n, double* y,
               double* dist) {
  double Q[9], M[9];
  bp_inv3(E, Q);
  bp_mat3_ata(Q, M);
  BpMetric mt;
  bp_metric_init(M, &mt);
  for (int j = 0; j < n; ++j) {
    double lo[3], hi[3], z[3];
    for (int k = 0; k < 3; ++k) { lo[k] = lb[3 * j + k] - p[k]; hi[k] = ub[3 * j + k] - p[k]; }
    int mask = bp_box_qp(mt, lo, hi, z);
    bp_box_point(p, lb + 3 * j, ub + 3 * j, z, mask, y + 3 * j);
    double zz[3] = {y[3 * j] - p[0], y[3 * j + 1] - p[1], y[3 * j + 2] - p[2]};
    double w[3];
    bp_mat3_vec(Q, zz, w);
    dist[j] = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  }
}

// closest points of n polytopes (rows [n,R,4] = a0 a1 a2 b, padded rows a = 0, b = 10) to p in the metric of
// E (q_inv): y[n,3], dist[n]; returns the number of empty polytopes
int hh_polytope_qp(const double* E, const double* p, const double* rows4, int n, int R, double* y, double* dist) {
  double Q[9], M[9];
  bp_inv3(E, Q);
  bp_mat3_ata(Q, M);
  BpPolyMetric pm;
  bp_poly_metric_init(M, &pm);
  int empty = 0;
  for (int j = 0; j < n; ++j) {
    struct R4 {
      const double* r;
      double a(int i, int k) const { return r[4 * i + k]; }
      double b(int i) const { return r[4 * i + 3]; }
    } rows{rows4 + (size_t)j * R * 4};
    if (!bp_polytope_qp(pm, rows, R, p, y + 3 * j)) { ++empty; dist[j] = -1.0; continue; }
    double zz[3] = {y[3 * j] - p[0], y[3 * j + 1] - p[1], y[3 * j + 2] - p[2]};
    double w[3];
    bp_mat3_vec(Q, zz, w);
    dist[j] = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  }
  return empty;
}

// closest points between the segment p0..p1 and n polytopes (rows4 as above), offsets shrunk by `shrink`
int hh_seg_polytope(const double* p0, const double* p1, const double* rows4, int n, int R, double shrink, double* x,
                    double* phi, double* dist2) {
  double d[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]};
  int empty = 0;
  for (int j = 0; j < n; ++j) {
    struct R4 {
      const double* r;
      double a(int i, int k) const { return r[4 * i + k]; }
      double b(int i) const { return r[4 * i + 3]; }
    } rows{rows4 + (size_t)j * R * 4};
    if (!bp_seg_polytope_qp(rows, R, shrink, p0, d, x + 3 * j, phi + j, dist2 + j)) ++empty;
  }
  return empty;
}

void hh_seg_box(const double* p0, const double* p1, const double* lb, const double* ub, int n, double* x,
                double* phi) {
  double d[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]};
  for (int j = 0; j < n; ++j) {
    double d2;
    phi[j] = bp_seg_box(p0, d, lb + 3 * j, ub + 3 * j, x + 3 * j, &d2);
  }
}

int hh_pair_lp(const double* A1, const double* b1, int m1, const double* A2, const double* b2, int m2, double tol,
               double* xout, int* iters) {
  HostRows r1{A1, b1}, r2{A2, b2};
  return bp_pair_feasible(r1, m1, r2, m2, tol, xout, iters);
}

int hh_pair_lp_t0(const double* A1, const double* b1, int m1, const double* A2, const double* b2, int m2, double tol,
                  double* xout, int* iters, double t0_scale) {
  HostRows r1{A1, b1}, r2{A2, b2};
  return bp_pair_feasible(r1, m1, r2, m2, tol, xout, iters, true, t0_scale);
}

void hh_fk(const double* q, int n, double* p_ee, double* p_col, double* T_ee, double* jac) {
  for (int i = 0; i < n; ++i)
    bp_fk_iiwa14(q + 7 * i, p_ee + 3 * i, p_col + 21 * i, T_ee ? T_ee + 16 * i : nullptr,
                 jac ? jac + 42 * i : nullptr);
}

void hh_fk_kin(const double* q, const double* dq, int n, double* T_ee, double* jac, double* djac) {
  for (int i = 0; i < n; ++i) {
    double pe[3], pc[21];
    bp_fk_iiwa14(q + 7 * i, pe, pc, T_ee + 16 * i, jac + 42 * i, dq + 7 * i, djac + 42 * i);
  }
}

double hh_min_eig(const double* A) { return bp_sym3_min_eig(A); }


// ---- the native lock-step planner driver (csrc/bp_planner.h) with every request kind answered by callbacks: the
// CPU tests plug the oracle in and compare with the Python planner (tests/util.py: run_native_with_oracle) ----
typedef int (*hh_cb_set)(int qid, const bpplan::SetReq* req, int n_nodes, const bpplan::Node* nodes, bpplan::SetAns* out);
typedef int (*hh_cb_edges)(int qid, int id_new, int n_nodes, const bpplan::Node* nodes, const int* has_target,
                           const double* xd, bpplan::EdgeAns* out);
typedef int (*hh_cb_project)(int qid, int id0, int id1, const double* xd, int n_nodes, const bpplan::Node* nodes,
                             bpplan::ProjAns* out);
typedef int (*hh_cb_path)(int qid, int n_nodes, const int* edge_off, const int* edge_dst, const double* edge_w,
                          int* path_out, int* path_len);
// reduce_ineqs of a given set (the start fallback's previous end set): fills out->m_red, Ar, br
typedef int (*hh_cb_reduce)(int qid, const bpplan::ReduceReq* req, bpplan::SetAns* out);

struct HhCallbackExecutor : bpplan::Executor {
  hh_cb_set cb_set; hh_cb_edges cb_edges; hh_cb_project cb_project; hh_cb_path cb_path; hh_cb_reduce cb_reduce;
  int n_lanes = 1;
  int lanes() const override { return n_lanes; }
  void commit_node(int, int, int, const bpplan::Node&) override {}
  int collect(int, bpplan::Round&) override { return 0; }
  int submit(int, bpplan::Round& r, const std::vector<bpplan::Query>& qs) override {
    for (size_t k = 0; k < r.sets.size(); ++k) {
      const bpplan::Query& q = qs[r.set_owner[k]];
      if (int rc = cb_set(q.qid, &r.sets[k], (int)q.nodes.size(), q.nodes.data(), &r.set_ans[k])) return rc;
    }
    for (size_t k = 0; k < r.edges.size(); ++k) {
      const bpplan::Query& q = qs[r.edge_owner[k]];
      if (int rc = cb_edges(q.qid, r.edges[k].id_new, (int)q.nodes.size(), q.nodes.data(),
                            r.edge_has_target.data() + r.edges[k].first_pair, r.edge_xd.data() + 3 * (size_t)r.edges[k].first_pair,
                            r.edge_ans.data() + r.edges[k].first_pair)) return rc;
    }
    size_t po = 0;
    for (size_t k = 0; k < r.proj_owner.size(); ++k) {
      const bpplan::Query& q = qs[r.proj_owner[k]];
      for (int e = 0; e < r.proj_count[k]; ++e, ++po)
        if (int rc = cb_project(q.qid, r.projs[po].id0, r.projs[po].id1, r.projs[po].xd, (int)q.nodes.size(),
                                q.nodes.data(), &r.proj_ans[po])) return rc;
    }
    for (size_t k = 0; k < r.paths.size(); ++k) {
      const int n0 = r.node_off[k];
      if (int rc = cb_path(r.paths[k].qid, r.paths[k].n_nodes, r.edge_off.data() + n0, r.edge_dst.data(), r.edge_w.data(),
                           r.path_out.data() + k * (size_t)bpplan::MAX_PATH, &r.path_len[k])) return rc;
    }
    for (size_t k = 0; k < r.reduces.size(); ++k)
      if (int rc = cb_reduce(r.reduces[k].qid, &r.reduces[k], &r.reduce_ans[k])) return rc;
    return 0;
  }
};

// the driver as bp_plan_run runs it: returns 3 (and err_msg[0] = the reason) when check_replan_inputs rejects the
// replanning inputs, before any callback runs
int hh_plan_batch(const bp_plan_in* in, bp_plan_out* out, hh_cb_set cb_set, hh_cb_edges cb_edges,
                  hh_cb_project cb_project, hh_cb_path cb_path, hh_cb_reduce cb_reduce, int lanes) {
  const std::string bad = bpplan::check_replan_inputs(*in);
  if (!bad.empty()) {
    std::snprintf(out->err_msg, 160, "%s", bad.c_str());
    return 3;
  }
  bpplan::Params par;
  std::vector<bpplan::Query> qs;
  bpplan::load_queries(*in, par, qs);
  HhCallbackExecutor ex;
  ex.cb_set = cb_set; ex.cb_edges = cb_edges; ex.cb_project = cb_project; ex.cb_path = cb_path; ex.cb_reduce = cb_reduce;
  ex.n_lanes = lanes > 0 ? lanes : 1;
  bpplan::RunStats st;
  std::vector<int> fin(qs.size(), -1);
  std::vector<double> fin_ms(qs.size(), -1.0);
  const int rc = bpplan::run_lockstep(qs, ex, par, &st, fin.data(), fin_ms.data());
  if (rc) return rc;
  bpplan::store_results(qs, st, fin.data(), fin_ms.data(), *out);
  return 0;
}

// numpy's PCG64 stream: n draws of rng.uniform(lo, hi, (n, 3)) from the given state
void hh_pcg64_uniform3(unsigned long long* state4, const double* lo, const double* hi, int n, double* out) {
  bpplan::Pcg64 g;
  g.set((const uint64_t*)state4);
  double range[3] = {hi[0] - lo[0], hi[1] - lo[1], hi[2] - lo[2]};
  g.uniform3(lo, range, n, out);
  g.get((uint64_t*)state4);
}

// sizes of the records the Python side mirrors with ctypes
int hh_sizeof(int what) {
  switch (what) {
    case 0: return (int)sizeof(bpplan::SetReq);
    case 1: return (int)sizeof(bpplan::SetAns);
    case 2: return (int)sizeof(bpplan::Node);
    case 3: return (int)sizeof(bpplan::EdgeAns);
    case 4: return (int)sizeof(bpplan::ProjAns);
    case 5: return (int)sizeof(bpplan::ReduceReq);
    case 6: return (int)sizeof(bp_plan_in);
    case 7: return (int)sizeof(bp_plan_out);
    default: return -1;
  }
}

}  // extern "C"
