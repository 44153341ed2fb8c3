// bp_planner.h -- native lock-step driver of the planner loop (host C++, no CUDA in this file).
//
// Restates, per query, the control flow of bound_planner/BoundPlanner/BoundPlanner.py:
//   plan_convex_set_path  :174-584   start / end sets (incl. the replanning branch :231-276 and the start-in-collision
//                                    fallbacks :296-324), sampling loop, dedupe, convergence test
//   compute_via_points    :586-743   with_rot=False branch (the via points are the p_proj's)
//   add_edges             :789-896   intersection nodes, projection points, edge costs (quirk Q6)
// as an explicit state machine (bpplan::Query) that emits REQUESTS for geometric primitives and is resumed with
// their answers -- the same protocol as the generator of boundplanner_b200/planner.py, which stays the readable
// statement of the loop and the thing this file is tested against (same paths, set sequences and via points).
// bpplan::run_lockstep advances all queries of a batch together: every round it collects the pending request of
// every live query, hands them to an Executor by KIND (one batched kernel chain per kind on the GPU executor of
// bpgeo.cu; callbacks into the test harness tests/host_harness.cpp), and resumes the queries.
// What is NOT here (as in planner.py): the final via-point NLP with rotations (Ipopt, :540-555).
#pragma once
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/bpgeo.h"

namespace bpplan {

constexpr int MAX_NODES = 64;     // graph nodes per query (2 + 20 samples + via-point re-samples)
constexpr int NODE_ROWS = 24;     // rows of a reduced node set (the reference's sets have at most 20)
constexpr int SET_ROWS = 48;      // BP_MAX_ROWS
constexpr int REF_MAX_ROWS = 20;  // the reference's MVIE buffers (quirk Q5)
constexpr int MAX_PATH = 64;
constexpr int FIT_SAMPLES = 20;   // check_intersection walks 20 rotations (:745-772)
constexpr int OBS_ROWS = 15;      // rows of a polytope obstacle (normalize_set_size, padded with a = 0, b = 10)
constexpr int MAX_PREV_SETS = 64; // previous sets per query (a planned sequence has at most MAX_PATH sets)

// error classes of the Python planner: RuntimeError / ValueError / IndexError / AttributeError
enum ErrKind { ERR_NONE = 0, ERR_RUNTIME = 1, ERR_VALUE = 2, ERR_INDEX = 3, ERR_ATTRIBUTE = 4 };

// ---- numpy's default generator (PCG64: 128-bit LCG, XSL-RR output), Generator.uniform's stream ----
struct Pcg64 {
  unsigned __int128 state, inc;
  void set(const uint64_t s[4]) {   // (state_hi, state_lo, inc_hi, inc_lo)
    state = ((unsigned __int128)s[0] << 64) | s[1];
    inc = ((unsigned __int128)s[2] << 64) | s[3];
  }
  void get(uint64_t s[4]) const {
    s[0] = (uint64_t)(state >> 64); s[1] = (uint64_t)state; s[2] = (uint64_t)(inc >> 64); s[3] = (uint64_t)inc;
  }
  uint64_t next64() {
    const unsigned __int128 mult = ((unsigned __int128)2549297995355413924ULL << 64) | 4865540595714422341ULL;
    state = state * mult + inc;
    const uint64_t hi = (uint64_t)(state >> 64), lo = (uint64_t)state;
    const uint64_t x = hi ^ lo;
    const unsigned rot = (unsigned)(state >> 122);
    return (x >> rot) | (x << ((-rot) & 63));
  }
  double next_double() { return (double)(next64() >> 11) * (1.0 / 9007199254740992.0); }
  // rng.uniform(lo, hi, (n, 3)) with array bounds: lo + (hi - lo) * u, element by element in C order
  void uniform3(const double* lo, const double* range, int n, double* out) {
    for (int i = 0; i < n; ++i)
      for (int k = 0; k < 3; ++k) out[3 * i + k] = lo[k] + range[k] * next_double();
  }
};

// ---- request / answer records (one pending request per live query and round) ----
enum ReqKind { REQ_NONE = 0, REQ_SET = 1, REQ_EDGES = 2, REQ_PROJECT = 3, REQ_PATH = 4, REQ_REDUCE = 5 };
enum SetKind { SET_POINT = 0, SET_LINE = 1, SET_SAMPLE = 2 };

struct SetReq {           // find_set_around_point / find_set_collision_avoidance / the sampling round
  int qid, kind, fixed_mid, optimize, with_dv, n_cand;
  double p0[3], p1[3];
  const double* cand;     // [n_cand,3] (SET_SAMPLE)
};
struct SetAns {
  int status, rows_peak, m, m_red, collision, first;
  double dv;
  double A[SET_ROWS * 3], b[SET_ROWS], Ar[SET_ROWS * 3], br[SET_ROWS], Q[9], P[3];
};
struct EdgeReq {          // set_intersection + check_intersection of node id_new against nodes 0 .. id_new-1
  int qid, id_new, n_others, first_pair;   // answers: pair first_pair + k  <->  (node k, id_new)
};
struct EdgeAns {          // proj: projection of the pair's target point onto the intersection (when ok and asked for)
  int ok, fits;
  double x[3], omega;
  int proj_ok;
  double proj[3];
};
struct ProjReq { int qid, id0, id1; double xd[3]; };     // projection onto rows(node id0) + rows(node id1)
struct ProjAns { double x[3]; int status; };
struct PathReq { int qid, n_nodes, edge_begin; };        // CSR of the query's intersection graph (see Round)
struct ReduceReq {        // reduce_ineqs of a given set (the previous end set of the start fallback, :318-327);
  int qid, m;             // answered in a SetAns (m_red, Ar, br)
  const double* rows;     // [m,4] (a0, a1, a2, b)
};

struct Node {             // graph node: reduced set + ellipsoid
  int m;
  double A[NODE_ROWS * 3], b[NODE_ROWS], Q[9], P[3], size;
  double c_size;          // tanh(0.25 - cbrt(size)): the node's factor in every edge cost (:876-878)
};
struct Inter {            // node of the intersection graph
  int id0, id1;
  bool conn_start, conn_end, has_proj, fits;
  double p_proj[3], p_via[4];
  std::vector<std::pair<int, double>> adj;   // (neighbour, weight) in insertion order (networkx's dict order)
};

struct Params {           // BoundPlanner.__init__ (:47-58)
  double obs_size_increase = 0.01, ws_min[3] = {-1.0, -1.0, 0.0}, ws_max[3] = {1.0, 1.0, 1.2};
  double w_size = 0.1, c_fit = 1.0, w_bias = 0.01;
  int max_iters = 20, nr_optimized = 10, max_samples = 500, sample_chunk = 32;
  int max_rounds = 4000;  // safety net of the lock-step loop (the reference's loop has none)
  int threads = 1;        // host threads that resume the state machines of a round (the queries are independent)
  int pool_min = 64;      // rounds with fewer live queries are resumed by the calling thread alone
};

struct QueryInput {
  const double* boxes;    // [n_obs,6] (lb, ub), uninflated; or NULL when obs_rows is set
  const double* obs_rows; // [n_obs,OBS_ROWS,4] (a0, a1, a2, b) of inflated polytope obstacles, or NULL
  int n_obs;
  double start[3], end[3], l_ee[3], l_ee_end[3];
  double ee_samples[FIT_SAMPLES * 3];    // Rodrigues(omega_hat, |omega| k/19) l_ee, k = 0..19
  uint64_t rng[4];
  int has_first_sample;
  double first_sample[3];
  // replanning (:231-276) and the previous sets (sets_via_prev of the reference, oldest first)
  int replanning, new_obs, n_horizon, n_prev;
  const double* p_horizon;  // [n_horizon,3]
  const int* prev_row_off;  // [n_prev+1] offsets into prev_rows (absolute)
  const double* prev_rows;  // [.,4] (a0, a1, a2, b)
};

// 3x3 determinant the way LAPACK's unblocked LU does it (np.linalg.det): partial pivoting, column scaled by the
// reciprocal of the pivot, rank-1 update
inline double det3_lu(const double* q) {
  double a[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) a[i][j] = q[3 * i + j];
  double det = 1.0;
  for (int j = 0; j < 3; ++j) {
    int p = j;
    for (int i = j + 1; i < 3; ++i)
      if (std::fabs(a[i][j]) > std::fabs(a[p][j])) p = i;
    if (a[p][j] == 0.0) return 0.0;
    if (p != j) {
      for (int k = 0; k < 3; ++k) std::swap(a[p][k], a[j][k]);
      det = -det;
    }
    const double r = 1.0 / a[j][j];
    for (int i = j + 1; i < 3; ++i) a[i][j] *= r;
    for (int i = j + 1; i < 3; ++i)
      for (int k = j + 1; k < 3; ++k) a[i][k] -= a[i][j] * a[j][k];
  }
  return det * a[0][0] * a[1][1] * a[2][2];
}

struct Query {
  // ---- program counter ----
  enum Pc { PC_START, PC_WAIT_START_SET, PC_WAIT_START_LINE, PC_WAIT_START_POINT, PC_WAIT_START_REDUCE,
            PC_WAIT_END_LINE, PC_EDGES_BEGIN, PC_WAIT_EDGES,
            PC_PROJECT_NEXT, PC_WAIT_PROJECT, PC_EDGES_DONE, PC_LOOP_TOP, PC_WAIT_PATH, PC_WAIT_SAMPLE,
            PC_SAMPLES_NEXT, PC_WAIT_SETPOINT, PC_DONE };
  enum After { AFTER_START_NODE, AFTER_END_NODE, AFTER_SAMPLE_NODE };

  int qid = 0;
  int scene = 0;              // the scene of the batch this query plans against (query_scene[qid], else qid)
  const Params* par = nullptr;
  QueryInput in;
  Pcg64 rng;
  Pc pc = PC_START;
  After after = AFTER_START_NODE;

  // pending request (exactly one kind when the query is live)
  int req_kind = REQ_NONE;
  SetReq set_req;
  EdgeReq edge_req;
  std::vector<ProjReq> proj_reqs;          // the projections of one add_edges call that are ready together
  // an "edges" request also carries, per other node v, the point that a hit (v, id_new) will be projected from:
  // it is known before the answers when v (or id_new) already has intersection nodes -- the first candidate of the
  // hit is then the oldest of those -- so that projection is computed in the same device round, gated by the hit
  std::vector<int> spec_target;            // [n_others] intersection node whose p_proj is the target, -1: none yet
  std::vector<double> spec_xd;             // [n_others,3]
  PathReq path_req;
  ReduceReq reduce_req;
  std::vector<double> cand;                // candidates of the pending sampling request

  // result
  int err_kind = ERR_NONE;
  std::string err_msg;
  bool finished = false;
  std::vector<int> path, set_ids;
  std::vector<double> p_via;               // [n,3]
  double p_horizon_max[3] = {0.0, 0.0, 0.0};   // the horizon point of a replanning query's start segment
  int rounds = 0;

  // planner state
  double start[3], end[3];
  std::vector<Node> nodes;
  std::vector<Inter> inter;
  std::vector<std::vector<int>> by_node;   // graph node -> its intersection nodes (ascending ids)
  bool connected = false, sampled_first = false, have_old = false;
  int nr_samples = 0, nr_sets = 0, nr_edges = 0, nr_inter_set = 0, j_iter = 0;
  std::vector<double> p_via_old, samples;  // samples: [n,3] of the current outer iteration
  int sample_idx = 0;
  bool have_pre = false;
  SetAns pre;
  int drawn = 0;
  Pcg64 rng_chunk_start;
  // add_edges in flight
  int e_id_new = 0;
  struct Hit { int vid, inter_id; bool fits; int target; bool pending; bool have_spec = false; double spec[3] = {0, 0, 0}; };
  std::vector<Hit> hits;
  size_t hit_next = 0;                     // first hit whose bookkeeping has not run yet
  size_t proj_first = 0, proj_end = 0;     // hits [proj_first, proj_end) have their projection in flight

  void fail(int kind, const std::string& msg) {
    err_kind = kind; err_msg = msg; finished = true; pc = PC_DONE; req_kind = REQ_NONE;
  }
  // planner._set_errors (ConvexSetFinder.py:438, :516)
  bool set_error(int status, int rows /* -1: None */) {
    char buf[160];
    if (status == 1) { fail(ERR_RUNTIME, "Ellipse violates constraints"); return true; }
    if (status == 2) { fail(ERR_VALUE, "convex set needs more rows than the kernels hold"); return true; }
    if (status == 5 || (status == 0 && rows > REF_MAX_ROWS)) {
      snprintf(buf, sizeof(buf), "could not broadcast input array from shape (%d,) into shape (%d,)", rows, REF_MAX_ROWS);
      fail(ERR_VALUE, buf);
      return true;
    }
    if (status == 3 || status == 4) {
      snprintf(buf, sizeof(buf), "MVIE failed (status %d)", status);
      fail(ERR_RUNTIME, buf);
      return true;
    }
    return false;
  }

  static double max_violation(const double* A, const double* b, int m, const double* x) {
    double v = -INFINITY;
    for (int i = 0; i < m; ++i) {
      const double s = A[3 * i] * x[0] + A[3 * i + 1] * x[1] + A[3 * i + 2] * x[2] - b[i];
      if (s > v) v = s;
    }
    return v;
  }

  // max over rows [m,4] of A x - b, formed as (a0 x0 + a1 x1) + a2 x2 - b without contraction (planner._rows_minus_b)
  static double max_rows_minus_b(const double* rows, int m, const double* x) {
    double v = -INFINITY;
    for (int i = 0; i < m; ++i) {
      const double* a = rows + 4 * i;
      const double s = (a[0] * x[0] + a[1] * x[1]) + a[2] * x[2] - a[3];
      if (s > v) v = s;
    }
    return v;
  }

  // :231-266 (SetSequencePlanner.replanning_horizon_index): how far along the horizon the previous sets still hold
  int horizon_index() const {
    int idx = 1;
    for (int s = 0; s < in.n_prev; ++s) {
      const double* rows = in.prev_rows + 4 * (size_t)in.prev_row_off[s];
      const int m = in.prev_row_off[s + 1] - in.prev_row_off[s];
      const bool start_in = max_rows_minus_b(rows, m, start) < 1e-8;
      int first_out = -1;
      for (int h = 0; h < in.n_horizon && first_out < 0; ++h)
        if (!(max_rows_minus_b(rows, m, in.p_horizon + 3 * (size_t)h) < 1e-8)) first_out = h;
      if (first_out >= 0) {
        if (first_out != 0 && start_in) idx = std::max(idx, first_out - 1);
      } else if (start_in) {
        idx = in.n_horizon - 1;
        break;
      }
    }
    if (in.new_obs) idx = 1;
    return idx;
  }

  // the new_obs fallback's test (:306-312, quirk Q12): `start` inside an inflated obstacle (no row with A x - b > 0;
  // polytopes: all 15 rows, boxes: the six box rows, as the push-out of `end` forms them)
  bool start_in_obstacle() const {
    const double r = par->obs_size_increase;
    for (int o = 0; o < in.n_obs; ++o) {
      bool any_pos = false;
      if (in.obs_rows) {
        const double* ro = in.obs_rows + (size_t)o * OBS_ROWS * 4;
        for (int i = 0; i < OBS_ROWS; ++i) {
          const double* a = ro + 4 * i;
          any_pos = any_pos || ((a[0] * start[0] + a[1] * start[1]) + a[2] * start[2] - a[3] > 0.0);
        }
      } else {
        const double* bx = in.boxes + 6 * o;
        for (int k = 0; k < 3; ++k)
          any_pos = any_pos || (start[k] - (bx[3 + k] + r) > 0.0) || (-start[k] - (-bx[k] + r) > 0.0);
      }
      if (!any_pos) return true;
    }
    return false;
  }

  void init(int id, const Params* p, const QueryInput& qi) {
    qid = id; par = p; in = qi;
    nodes.reserve(MAX_NODES); by_node.reserve(MAX_NODES); inter.reserve(128); hits.reserve(MAX_NODES);
    cand.reserve(3 * 64); cand_tmp.reserve(128); spec_target.reserve(MAX_NODES); spec_xd.reserve(3 * MAX_NODES);
    rng.set(qi.rng);
    for (int k = 0; k < 3; ++k) { start[k] = qi.start[k]; end[k] = qi.end[k]; }
    // :199-204, obstacle by obstacle in order: an `end` inside an inflated obstacle is pushed out through the
    // face of largest A x - b (rows [I; -I], b = [ub + r, -lb + r], padded rows -10)
    const double r = par->obs_size_increase;
    if (qi.obs_rows) {
      // general polytopes: all 15 rows, padding (0, 0, 0, 10) included.  A x - b is formed as (a0 x0 + a1 x1) + a2 x2
      // - b without contraction, as the Python planner's general path does: this differs from the reference's
      // ob[0] @ end (BLAS, may fuse) in the last bits only, and is exact for box rows (+-e_k), where it equals the
      // box arithmetic below
      for (int o = 0; o < qi.n_obs; ++o) {
        const double* ro = qi.obs_rows + (size_t)o * OBS_ROWS * 4;
        double viol[OBS_ROWS];
        bool any_pos = false;
        for (int i = 0; i < OBS_ROWS; ++i) {
          const double* a = ro + 4 * i;
          viol[i] = (a[0] * end[0] + a[1] * end[1]) + a[2] * end[2] - a[3];
          any_pos = any_pos || (viol[i] > 0.0);
        }
        if (any_pos) continue;
        int idx = 0;                                             // first index of the maximum (np.argmax)
        for (int i = 1; i < OBS_ROWS; ++i)
          if (viol[i] > viol[idx]) idx = i;
        const double step = viol[idx] - r;
        for (int k = 0; k < 3; ++k) end[k] -= step * ro[4 * idx + k];
      }
      return;
    }
    for (int o = 0; o < qi.n_obs; ++o) {
      const double* bx = qi.boxes + 6 * o;
      double viol[6];
      bool any_pos = false;
      for (int k = 0; k < 3; ++k) {
        viol[k] = end[k] - (bx[3 + k] + r);
        viol[3 + k] = -end[k] - (-bx[k] + r);
      }
      for (int k = 0; k < 6; ++k) any_pos = any_pos || (viol[k] > 0.0);
      if (any_pos) continue;
      int idx = 0;
      for (int k = 1; k < 6; ++k)
        if (viol[k] > viol[idx]) idx = k;
      if (!(viol[idx] > -10.0)) idx = 6;                       // a padded row wins the argmax: zero normal, no move
      if (idx < 6) {
        const double sgn = idx < 3 ? 1.0 : -1.0;
        end[idx % 3] -= (viol[idx] - r) * sgn;
      }
    }
  }

  // ---- graph bookkeeping ----
  bool add_node(const double* Ar, const double* br, int m_red, const double* Q, const double* P) {
    if ((int)nodes.size() >= MAX_NODES) {
      fail(ERR_VALUE, "more than 64 graph nodes in one query");
      return false;
    }
    if (m_red > NODE_ROWS) {
      fail(ERR_VALUE, "graph node with more than 24 rows");
      return false;
    }
    Node n;
    n.m = m_red;
    std::memset(n.A, 0, sizeof(n.A));
    for (int i = 0; i < NODE_ROWS; ++i) n.b[i] = 10.0;
    std::memcpy(n.A, Ar, sizeof(double) * 3 * m_red);
    std::memcpy(n.b, br, sizeof(double) * m_red);
    std::memcpy(n.Q, Q, sizeof(n.Q));
    std::memcpy(n.P, P, sizeof(n.P));
    n.size = 1.0 / det3_lu(Q);
    n.c_size = std::tanh(0.25 - std::cbrt(n.size));
    nodes.push_back(n);
    by_node.emplace_back();
    nr_sets += 1;
    return true;
  }
  int add_inter(int id0, int id1, bool cs, bool ce, const double* p_proj, const double* via, bool fits) {
    Inter it;
    it.id0 = id0; it.id1 = id1; it.conn_start = cs; it.conn_end = ce; it.fits = fits;
    it.has_proj = p_proj != nullptr;
    for (int k = 0; k < 3; ++k) it.p_proj[k] = p_proj ? p_proj[k] : 0.0;
    for (int k = 0; k < 4; ++k) it.p_via[k] = via ? via[k] : 0.0;
    inter.push_back(std::move(it));
    return (int)inter.size() - 1;
  }

  // candidates of one hit: the intersection nodes that share vid or id_new, ascending, without `me`
  void edge_candidates(int vid, int id_new, int me, std::vector<int>& out) const {
    out.clear();
    const std::vector<int>& a = by_node[vid];
    const std::vector<int>& b = by_node[id_new];
    size_t i = 0, j = 0;
    while (i < a.size() || j < b.size()) {
      int v;
      if (j >= b.size() || (i < a.size() && a[i] <= b[j])) { v = a[i]; if (j < b.size() && b[j] == v) ++j; ++i; }
      else { v = b[j]; ++j; }
      if (v != me) out.push_back(v);
    }
  }

  // ---- add_edges (:789-896) as a sub-machine: PC_EDGES_BEGIN .. PC_EDGES_DONE ----
  void edges_begin(int id_new, After a) {
    e_id_new = id_new; after = a;
    hits.clear(); hit_next = 0; proj_first = proj_end = 0;
    edges_connected = false;
    pc = PC_EDGES_BEGIN;
  }
  bool edges_connected = false;
  std::vector<int> cand_tmp;

  // the projection target of a hit: p_proj of the first candidate (or `end` when that node has none); -2: the hit
  // has no candidate at all (no edge, no projection), -1: use `end`
  int projection_target(const Hit& h) {
    edge_candidates(h.vid, e_id_new, h.inter_id, cand_tmp);
    if (cand_tmp.empty()) return -2;
    return cand_tmp[0];
  }

  // bookkeeping of hit h once its projection (if any) is known: edges, connection flags, costs
  void hit_bookkeeping(const Hit& h) {
    Inter& me = inter[h.inter_id];
    edge_candidates(h.vid, e_id_new, h.inter_id, cand_tmp);
    for (int eid : cand_tmp) {
      Inter& ed = inter[eid];
      const bool cond1 = ed.id0 == h.vid || ed.id1 == h.vid;
      const double c_size = cond1 ? nodes[h.vid].c_size : nodes[e_id_new].c_size;
      nr_edges += 2;
      const double* pp = ed.has_proj ? ed.p_proj : end;
      const double d0 = me.p_proj[0] - pp[0], d1 = me.p_proj[1] - pp[1], d2 = me.p_proj[2] - pp[2];
      const double dist = std::sqrt(d0 * d0 + d1 * d1 + d2 * d2);
      const bool cs = me.conn_start || ed.conn_start, ce = me.conn_end || ed.conn_end;
      me.conn_start = ed.conn_start = cs;
      me.conn_end = ed.conn_end = ce;
      edges_connected = cs && ce;                                 // last edge wins (quirk Q6)
      double cost = dist * (1 + par->w_size * c_size) + par->w_bias;
      if (!h.fits) cost += par->c_fit;
      me.adj.emplace_back(eid, cost);
      ed.adj.emplace_back(h.inter_id, cost);
    }
  }

  // ---- compute_via_points (:586-743, with_rot=False) ----
  bool via_points(const std::vector<int>& pth, std::vector<double>& pv, std::vector<int>& seq_via) {
    const int n = (int)pth.size();
    std::vector<int> seq(n);
    int last_id = 0;
    for (int i = 0; i < n; ++i) {
      const Inter& nd = inter[pth[i]];
      if (i == 0) last_id = nd.id0;
      else if (nd.id0 != last_id) last_id = nd.id0;
      else if (nd.id1 != last_id) last_id = nd.id1;
      seq[i] = last_id;
    }
    pv.assign(start, start + 3);
    seq_via.clear();
    for (int i = 0; i + 2 < n; ++i) {
      const Inter& nd = inter[pth[1 + i]];
      if (!nd.has_proj) {
        // an intersection node without edges at its creation never got a projection point; on a path the
        // reference's x0 = np.concatenate((x0, None, [0.5])) (:595) raises this ValueError
        fail(ERR_VALUE, "all the input arrays must have same number of dimensions, but the array at index 0 has 1 "
                        "dimension(s) and the array at index 1 has 0 dimension(s)");
        return false;
      }
      const double* last = &pv[pv.size() - 3];
      const double d0 = nd.p_proj[0] - last[0], d1 = nd.p_proj[1] - last[1], d2 = nd.p_proj[2] - last[2];
      if (std::sqrt(d0 * d0 + d1 * d1 + d2 * d2) > 1e-4) {
        pv.insert(pv.end(), nd.p_proj, nd.p_proj + 3);
        seq_via.push_back(seq[i]);
      }
    }
    pv.insert(pv.end(), end, end + 3);
    seq_via.push_back(seq[n - 1]);
    return true;
  }

  void emit_set(int kind, const double* p0, const double* p1, int fixed_mid, int optimize, int with_dv) {
    req_kind = REQ_SET;
    set_req.qid = qid; set_req.kind = kind; set_req.fixed_mid = fixed_mid; set_req.optimize = optimize;
    set_req.with_dv = with_dv; set_req.n_cand = 0; set_req.cand = nullptr;
    for (int k = 0; k < 3; ++k) { set_req.p0[k] = p0[k]; set_req.p1[k] = p1 ? p1[k] : 0.0; }
  }
  void emit_sample_chunk() {
    const int c = std::min(par->sample_chunk, par->max_samples + 1 - drawn);
    double range[3];
    for (int k = 0; k < 3; ++k) range[k] = par->ws_max[k] - par->ws_min[k];
    rng_chunk_start = rng;
    cand.resize(3 * (size_t)c);
    rng.uniform3(par->ws_min, range, c, cand.data());
    req_kind = REQ_SET;
    set_req.qid = qid; set_req.kind = SET_SAMPLE; set_req.fixed_mid = 1;
    set_req.optimize = !(nr_samples + 1 >= par->nr_optimized);
    set_req.with_dv = 1; set_req.n_cand = c; set_req.cand = cand.data();
    for (int k = 0; k < 3; ++k) set_req.p0[k] = set_req.p1[k] = 0.0;
    pc = PC_WAIT_SAMPLE;
  }

  // Resume with the answer(s) to the pending request; returns when the next request is pending or the query is
  // finished.  set_ans / edge_ans (the n_others answers of this query) / proj_ans (one per pending projection) /
  // path_ans (node ids, len; len <= 0: no path).
  void resume(const SetAns* set_ans, const EdgeAns* edge_ans, const ProjAns* proj_ans, const int* path_ans, int path_len) {
    req_kind = REQ_NONE;
    for (;;) {
      switch (pc) {
        case PC_START: {
          if (in.replanning) {                                                            // :231-276
            int idx = horizon_index();
            const int H = in.n_horizon;
            if (idx < -H || idx >= H) {                  // self.p_horizon[idx] of a horizon too short
              char buf[96];
              snprintf(buf, sizeof(buf), "index %d is out of bounds for axis 0 with size %d", idx, H);
              fail(ERR_INDEX, buf);
              return;
            }
            if (idx < 0) idx += H;
            for (int k = 0; k < 3; ++k) p_horizon_max[k] = in.p_horizon[3 * (size_t)idx + k];
            emit_set(SET_LINE, start, p_horizon_max, 0, 0, 0);
            pc = PC_WAIT_START_LINE;
            return;
          }
          emit_set(SET_POINT, start, nullptr, 1, 1, 0);                                  // :278-283
          pc = PC_WAIT_START_SET;
          return;
        }
        case PC_WAIT_START_SET: {
          const SetAns& a = *set_ans;
          if (set_error(a.status, a.rows_peak)) return;
          double tip[3] = {start[0] + in.l_ee[0], start[1] + in.l_ee[1], start[2] + in.l_ee[2]};
          if (max_violation(a.A, a.b, a.m, tip) > 1e-8) {
            emit_set(SET_LINE, start, tip, 0, 0, 0);
            pc = PC_WAIT_START_LINE;
            return;
          }
          if (!add_node(a.Ar, a.br, a.m_red, a.Q, a.P)) return;
          pc = PC_EDGES_BEGIN;
          after_start_node();
          continue;
        }
        case PC_WAIT_START_LINE: {
          const SetAns& a = *set_ans;
          if (set_error(a.status, a.m)) return;
          if (a.collision) {                                                              // :296-324
            if (in.new_obs) {
              // the reference pushes `start` out of every inflated obstacle that contains it through `ob.A()` on a
              // list: AttributeError as soon as one does (quirk Q12); otherwise a start set around `start`
              if (start_in_obstacle()) { fail(ERR_ATTRIBUTE, "'list' object has no attribute 'A'"); return; }
              emit_set(SET_POINT, start, nullptr, 1, 1, 0);
              pc = PC_WAIT_START_POINT;
              return;
            }
            // "Could not find start set, reusing old end set": sets_via_prev[-1], IndexError on a first plan
            if (in.n_prev == 0) { fail(ERR_INDEX, "list index out of range"); return; }
            const int s = in.n_prev - 1;
            req_kind = REQ_REDUCE;
            reduce_req.qid = qid;
            reduce_req.m = in.prev_row_off[s + 1] - in.prev_row_off[s];
            reduce_req.rows = in.prev_rows + 4 * (size_t)in.prev_row_off[s];
            pc = PC_WAIT_START_REDUCE;
            return;
          }
          if (!add_node(a.Ar, a.br, a.m_red, a.Q, a.P)) return;
          after_start_node();
          continue;
        }
        case PC_WAIT_START_POINT: {                     // new_obs start set around `start` (no tool-tip test)
          const SetAns& a = *set_ans;
          if (set_error(a.status, a.rows_peak)) return;
          if (!add_node(a.Ar, a.br, a.m_red, a.Q, a.P)) return;
          after_start_node();
          continue;
        }
        case PC_WAIT_START_REDUCE: {                    // the reused end set: q_ellipse = I, p_mid = start
          const double eye[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
          if (!add_node(set_ans->Ar, set_ans->br, set_ans->m_red, eye, start)) return;
          after_start_node();
          continue;
        }
        case PC_WAIT_END_LINE: {                                                          // :381-390
          const SetAns& a = *set_ans;
          if (set_error(a.status, a.m)) return;
          if (!add_node(a.Ar, a.br, a.m_red, a.Q, a.P)) return;
          double via[4] = {end[0], end[1], end[2], 1.0};
          const int id = add_inter(1, 1, false, true, end, via, true);
          by_node[1].push_back(id);
          edges_begin(1, AFTER_END_NODE);
          continue;
        }
        case PC_EDGES_BEGIN: {
          if (e_id_new == 0) { pc = PC_EDGES_DONE; continue; }       // no other node yet
          req_kind = REQ_EDGES;
          edge_req.qid = qid; edge_req.id_new = e_id_new; edge_req.n_others = e_id_new; edge_req.first_pair = 0;
          spec_target.assign((size_t)e_id_new, -1);
          spec_xd.assign(3 * (size_t)e_id_new, 0.0);
          for (int v = 0; v < e_id_new; ++v) {
            int t = -1;
            if (!by_node[v].empty()) t = by_node[v][0];
            if (!by_node[e_id_new].empty() && (t < 0 || by_node[e_id_new][0] < t)) t = by_node[e_id_new][0];
            spec_target[(size_t)v] = t;
            if (t >= 0) {
              const double* xd = inter[t].has_proj ? inter[t].p_proj : end;
              for (int c = 0; c < 3; ++c) spec_xd[3 * (size_t)v + c] = xd[c];
            }
          }
          pc = PC_WAIT_EDGES;
          return;
        }
        case PC_WAIT_EDGES: {
          for (int v = 0; v < e_id_new; ++v) {
            const EdgeAns& ea = edge_ans[v];
            if (!ea.ok) continue;
            double via[4] = {ea.x[0], ea.x[1], ea.x[2], ea.fits ? ea.omega : 0.0};
            const int id = add_inter(v, e_id_new, false, false, nullptr, via, ea.fits != 0);
            nr_inter_set += 2;
            hits.push_back(Hit{v, id, ea.fits != 0, -2, false});
            if (spec_target[(size_t)v] >= 0 && ea.proj_ok) {          // projected in this very round
              Hit& h = hits.back();
              h.have_spec = true;
              for (int c = 0; c < 3; ++c) h.spec[c] = ea.proj[c];
            }
          }
          // the reference registers a hit in the node index when it is created, hit by hit; the candidates of hit
          // k therefore never contain the hits after it: by_node is filled as the hits are processed
          hit_next = 0;
          pc = PC_PROJECT_NEXT;
          continue;
        }
        case PC_PROJECT_NEXT: {
          // process the hits in order; the projections whose target point is already known go out together
          proj_reqs.clear();
          proj_first = hit_next;
          size_t k = hit_next;
          // register + resolve targets for as many hits as possible
          while (k < hits.size()) {
            Hit& h = hits[k];
            by_node[h.vid].push_back(h.inter_id);
            by_node[e_id_new].push_back(h.inter_id);
            h.target = projection_target(h);
            bool depends_on_pending = false;
            if (h.target >= 0) {
              for (size_t q = proj_first; q < k; ++q)
                if (hits[q].inter_id == h.target && hits[q].pending) depends_on_pending = true;
            }
            if (depends_on_pending) {            // its target is a projection of this very batch: next round
              by_node[h.vid].pop_back();
              by_node[e_id_new].pop_back();
              break;
            }
            h.pending = h.target != -2;
            if (h.pending && h.have_spec && h.target == spec_target[(size_t)h.vid]) {
              Inter& me = inter[h.inter_id];                        // already projected with the edges request
              for (int c = 0; c < 3; ++c) me.p_proj[c] = h.spec[c];
              me.has_proj = true;
              h.pending = false;
            }
            if (h.pending) {
              ProjReq pr;
              pr.qid = qid; pr.id0 = h.vid; pr.id1 = e_id_new;
              const Inter* t = h.target >= 0 ? &inter[h.target] : nullptr;
              const double* xd = (t && t->has_proj) ? t->p_proj : end;
              for (int c = 0; c < 3; ++c) pr.xd[c] = xd[c];
              proj_reqs.push_back(pr);
            }
            ++k;
          }
          proj_end = k;
          if (proj_end == proj_first) { pc = PC_EDGES_DONE; continue; }      // no hits (left)
          if (proj_reqs.empty()) {                  // nothing left to ask for: the bookkeeping of these hits runs now
            proj_ans = nullptr;
            pc = PC_WAIT_PROJECT;
            continue;
          }
          req_kind = REQ_PROJECT;
          pc = PC_WAIT_PROJECT;
          return;
        }
        case PC_WAIT_PROJECT: {
          // the bookkeeping needs by_node as it was when each hit was created: rebuild it incrementally
          // (un-register the hits of this batch, then replay them one by one)
          for (size_t k = proj_end; k-- > proj_first;) {
            by_node[hits[k].vid].pop_back();
            by_node[e_id_new].pop_back();
          }
          size_t pi = 0;
          for (size_t k = proj_first; k < proj_end; ++k) {
            Hit& h = hits[k];
            by_node[h.vid].push_back(h.inter_id);
            by_node[e_id_new].push_back(h.inter_id);
            if (h.pending) {
              Inter& me = inter[h.inter_id];
              for (int c = 0; c < 3; ++c) me.p_proj[c] = proj_ans[pi].x[c];
              me.has_proj = true;
              ++pi;
              h.pending = false;
            }
            hit_bookkeeping(h);
          }
          hit_next = proj_end;
          pc = hit_next < hits.size() ? PC_PROJECT_NEXT : PC_EDGES_DONE;
          continue;
        }
        case PC_EDGES_DONE: {
          const bool conn = edges_connected;
          if (after == AFTER_START_NODE) {
            connected = conn;
            // :361-375: end (and its tool tip) already inside the start set
            const Node& n0 = nodes[0];
            double tip[3] = {end[0] + in.l_ee_end[0], end[1] + in.l_ee_end[1], end[2] + in.l_ee_end[2]};
            if (max_violation(n0.A, n0.b, n0.m, end) < 1e-8 && max_violation(n0.A, n0.b, n0.m, tip) < 1e-8) {
              path.assign(1, 0);
              set_ids.assign(1, 0);
              p_via.assign(start, start + 3);
              p_via.insert(p_via.end(), end, end + 3);
              finished = true; pc = PC_DONE;
              return;
            }
            emit_set(SET_LINE, end, tip, 0, 0, 0);
            pc = PC_WAIT_END_LINE;
            return;
          }
          connected = conn || connected;
          if (after == AFTER_END_NODE) { pc = PC_LOOP_TOP; continue; }
          pc = PC_SAMPLES_NEXT;
          continue;
        }
        case PC_LOOP_TOP: {                                                               // :430-534
          have_pre = false;
          if (connected) {
            req_kind = REQ_PATH;
            path_req.qid = qid; path_req.n_nodes = (int)inter.size(); path_req.edge_begin = 0;
            pc = PC_WAIT_PATH;
            return;
          }
          if (!sampled_first && in.has_first_sample) {
            samples.assign(in.first_sample, in.first_sample + 3);
            sample_idx = 0;
            pc = PC_SAMPLES_NEXT;
            continue;
          }
          drawn = 0;
          emit_sample_chunk();
          return;
        }
        case PC_WAIT_PATH: {
          if (path_len <= 0 || path_len > MAX_PATH) {
            fail(ERR_RUNTIME, path_len <= 0 ? "No path between 0 and 1." : "shortest path longer than 64 nodes");
            return;
          }
          path.assign(path_ans, path_ans + path_len);
          std::vector<double> pv;
          std::vector<int> seq_via;
          if (!via_points(path, pv, seq_via)) return;
          bool same = have_old && p_via_old.size() == pv.size();
          if (same) {
            double s = 0.0;
            for (size_t i = 0; i < pv.size(); ++i) { const double d = p_via_old[i] - pv[i]; s += d * d; }
            same = std::sqrt(s) < 1e-4;
          }
          p_via = pv;
          set_ids = seq_via;
          if (same) { finished = true; pc = PC_DONE; return; }                          // "Found path solution"
          samples.assign(pv.begin() + 3, pv.end() - 3);
          p_via_old = pv;
          have_old = true;
          sample_idx = 0;
          pc = PC_SAMPLES_NEXT;
          continue;
        }
        case PC_WAIT_SAMPLE: {
          const SetAns& a = *set_ans;
          const int c = set_req.n_cand;
          if (a.first < 0 || a.first >= c) {
            drawn += c;
            if (drawn < par->max_samples + 1) { emit_sample_chunk(); return; }
            fail(ERR_RUNTIME, "(PosPath) Could not find collision-free sample");          // :477-478
            return;
          }
          const int n = drawn + a.first + 1;
          // the reference's one-at-a-time loop consumed exactly n draws
          rng = rng_chunk_start;
          for (int i = 0; i < 3 * (a.first + 1); ++i) rng.next64();
          if (n >= par->max_samples) { fail(ERR_RUNTIME, "(PosPath) Could not find collision-free sample"); return; }
          nr_samples += 1;
          if (nr_samples > par->max_iters) { fail(ERR_RUNTIME, "(PosPath) Exceeded max iterations"); return; }
          samples.assign(cand.begin() + 3 * a.first, cand.begin() + 3 * a.first + 3);
          pre = a;
          have_pre = true;
          sample_idx = 0;
          pc = PC_SAMPLES_NEXT;
          continue;
        }
        case PC_SAMPLES_NEXT: {
          if (3 * (size_t)sample_idx >= samples.size()) { pc = PC_LOOP_TOP; continue; }
          j_iter += 1;
          const int optimize = !(nr_samples >= par->nr_optimized);
          if (have_pre) { set_ans = &pre; pc = PC_WAIT_SETPOINT; continue; }
          emit_set(SET_POINT, &samples[3 * (size_t)sample_idx], nullptr, 1, optimize, 1);
          pc = PC_WAIT_SETPOINT;
          return;
        }
        case PC_WAIT_SETPOINT: {
          const SetAns& a = *set_ans;
          const int optimize = have_pre ? set_req.optimize : !(nr_samples >= par->nr_optimized);
          if (set_error(a.status, optimize ? a.rows_peak : -1)) return;
          sampled_first = true;
          sample_idx += 1;
          if (a.dv > 0.01) {                                                              // :505-512
            if (!add_node(a.Ar, a.br, a.m_red, a.Q, a.P)) return;
            edges_begin((int)nodes.size() - 1, AFTER_SAMPLE_NODE);
            continue;
          }
          pc = PC_SAMPLES_NEXT;
          continue;
        }
        case PC_DONE:
          return;
      }
    }
  }

  void after_start_node() {
    double via[4] = {start[0], start[1], start[2], 0.0};
    const int id = add_inter(0, 0, true, false, start, via, true);
    by_node[0].push_back(id);
    edges_begin(0, AFTER_START_NODE);
  }
};

// ---- one lock-step round: the pending requests of all live queries, by kind ----
struct Round {
  std::vector<SetReq> sets;          std::vector<SetAns> set_ans;
  std::vector<EdgeReq> edges;        std::vector<EdgeAns> edge_ans;      // flat, EdgeReq::first_pair indexes it
  std::vector<int> edge_has_target;  std::vector<double> edge_xd;        // per pair: project this point when it hits
  std::vector<ProjReq> projs;        std::vector<ProjAns> proj_ans;
  std::vector<PathReq> paths;                                            // CSR over all graphs of the round:
  std::vector<int> node_off, edge_off, edge_dst;                         //   node_off[g], edge_off[node], edge_dst
  std::vector<double> edge_w;
  std::vector<int> path_out, path_len;                                   // [G, MAX_PATH], [G]
  std::vector<ReduceReq> reduces;    std::vector<SetAns> reduce_ans;     // answers: m_red, Ar, br
  std::vector<int> set_owner, edge_owner, proj_owner, proj_count, path_owner, reduce_owner;   // index into the query array
  void clear() {
    reduces.clear(); reduce_owner.clear();
    sets.clear(); edges.clear(); projs.clear(); paths.clear(); node_off.clear(); edge_off.clear(); edge_dst.clear();
    edge_has_target.clear(); edge_xd.clear();
    edge_w.clear(); set_owner.clear(); edge_owner.clear(); proj_owner.clear(); proj_count.clear(); path_owner.clear();
  }
};

// A small pool of host threads for the one loop of the driver that is worth it: resuming the (independent) state
// machines of a round.  parallel_for(n, fn) runs fn(i) for i in [0, n) on the pool and the calling thread.
struct HostPool {
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  const std::function<void(size_t)>* job = nullptr;
  size_t n_items = 0;
  std::atomic<size_t> next{0};
  int generation = 0, busy = 0;
  bool stop = false;

  explicit HostPool(int threads) {
    for (int t = 1; t < threads; ++t) workers.emplace_back([this] { loop(); });
  }
  ~HostPool() {
    { std::lock_guard<std::mutex> lk(mu); stop = true; }
    cv_work.notify_all();
    for (auto& w : workers) w.join();
  }
  void drain() {
    for (;;) {
      const size_t i = next.fetch_add(16);
      if (i >= n_items) break;
      const size_t e = std::min(n_items, i + 16);
      for (size_t k = i; k < e; ++k) (*job)(k);
    }
  }
  void loop() {
    int seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu);
        cv_work.wait(lk, [&] { return stop || generation != seen; });
        if (stop) return;
        seen = generation;
      }
      drain();
      {
        std::lock_guard<std::mutex> lk(mu);
        if (--busy == 0) cv_done.notify_one();
      }
    }
  }
  size_t min_items = 64;
  void parallel_for(size_t n, const std::function<void(size_t)>& fn) {
    if (workers.empty() || n < min_items) {
      for (size_t i = 0; i < n; ++i) fn(i);
      return;
    }
    {
      std::lock_guard<std::mutex> lk(mu);
      job = &fn; n_items = n; next.store(0); busy = (int)workers.size(); ++generation;
    }
    cv_work.notify_all();
    drain();
    std::unique_lock<std::mutex> lk(mu);
    cv_done.wait(lk, [&] { return busy == 0; });
  }
};

struct Executor {
  virtual ~Executor() {}
  // independent lock-step groups ("lanes") the executor can keep in flight at once: while one lane's round runs on
  // the device the host resumes and packs another (1: plain lock step)
  virtual int lanes() const { return 1; }
  // a node was added to query qid's graph (the executor keeps the tables the requests refer to)
  virtual void commit_node(int lane, int qid, int node_id, const Node& n) = 0;
  // start answering every request of the round (asynchronously, if the executor can) / wait for the answers
  // (set_ans / edge_ans / proj_ans / path_out / path_len / reduce_ans filled).  queries: for executors that look at the
  // planners' state (the test harness).  Return 0, or an error code that aborts the run.
  virtual int submit(int lane, Round& r, const std::vector<Query>& queries) = 0;
  virtual int collect(int lane, Round& r) = 0;
};

struct RunStats {
  int rounds = 0;                     // lock-step rounds of the longest lane
  long long set_requests = 0, edge_pairs = 0, projections = 0, paths = 0;
  double gather_ms = 0.0, resume_ms = 0.0;   // host time: building the rounds / resuming the state machines
};

// Advance all queries until every one is finished.  The queries are dealt to the executor's lanes (query i -> lane
// i mod L); every lane is a lock-step group of its own: each of its rounds collects the pending request of every
// live query of the lane, hands them to the executor and resumes the queries with the answers.  finish_round[q]
// (or null) receives the round of its lane in which query q finished, finish_ms[q] (or null) the wall time since
// the start of the run at that moment.
inline int run_lockstep(std::vector<Query>& qs, Executor& ex, const Params& par, RunStats* stats, int* finish_round,
                        double* finish_ms = nullptr) {
  const int L = std::max(1, std::min(ex.lanes(), (int)qs.size()));
  std::vector<Round> rounds_(L);
  std::vector<int> n_rounds(L, 0);
  std::vector<char> in_flight(L, 0);
  std::vector<size_t> committed(qs.size(), 0);
  const auto t_start = std::chrono::steady_clock::now();
  auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
  for (auto& q : qs) q.resume(nullptr, nullptr, nullptr, nullptr, 0);

  // gather the pending requests of lane l into its round and submit it; returns the number of live queries (or < 0)
  auto launch = [&](int l) -> int {
    const double t_g0 = now_ms();
    Round& r = rounds_[l];
    r.clear();
    size_t live = 0;
    for (size_t i = (size_t)l; i < qs.size(); i += (size_t)L) {
      Query& q = qs[i];
      // nodes added since the last round go to the executor's tables first
      for (; committed[i] < q.nodes.size(); ++committed[i]) ex.commit_node(l, q.qid, (int)committed[i], q.nodes[committed[i]]);
      if (q.finished) {
        if (finish_round && finish_round[i] < 0) finish_round[i] = n_rounds[l];
        if (finish_ms && finish_ms[i] < 0.0) finish_ms[i] = now_ms();
        continue;
      }
      ++live;
      switch (q.req_kind) {
        case REQ_SET: r.sets.push_back(q.set_req); r.set_owner.push_back((int)i); break;
        case REQ_EDGES: {
          EdgeReq e = q.edge_req;
          e.first_pair = (int)r.edge_has_target.size();
          r.edges.push_back(e); r.edge_owner.push_back((int)i);
          for (int v = 0; v < e.n_others; ++v) r.edge_has_target.push_back(q.spec_target[(size_t)v] >= 0 ? 1 : 0);
          r.edge_xd.insert(r.edge_xd.end(), q.spec_xd.begin(), q.spec_xd.end());
          break;
        }
        case REQ_PROJECT:
          r.proj_owner.push_back((int)i); r.proj_count.push_back((int)q.proj_reqs.size());
          r.projs.insert(r.projs.end(), q.proj_reqs.begin(), q.proj_reqs.end());
          break;
        case REQ_PATH: {
          PathReq p = q.path_req;
          p.edge_begin = (int)r.edge_dst.size();
          r.node_off.push_back(r.paths.empty() ? 0 : r.node_off.back() + r.paths.back().n_nodes);
          for (const Inter& it : q.inter) {
            r.edge_off.push_back((int)r.edge_dst.size());
            for (const auto& e : it.adj) { r.edge_dst.push_back(e.first); r.edge_w.push_back(e.second); }
          }
          r.paths.push_back(p); r.path_owner.push_back((int)i);
          break;
        }
        case REQ_REDUCE: r.reduces.push_back(q.reduce_req); r.reduce_owner.push_back((int)i); break;
        default:
          q.fail(ERR_RUNTIME, "planner state machine without a pending request");
          --live;
          break;
      }
    }
    if (live == 0) return 0;
    if (!r.paths.empty()) {
      r.node_off.push_back(r.node_off.back() + r.paths.back().n_nodes);
      r.edge_off.push_back((int)r.edge_dst.size());
    }
    ++n_rounds[l];
    if (n_rounds[l] > par.max_rounds) {
      for (size_t i = (size_t)l; i < qs.size(); i += (size_t)L)
        if (!qs[i].finished) qs[i].fail(ERR_RUNTIME, "lock-step round limit reached");
      return 0;
    }
    if (r.set_ans.size() < r.sets.size()) r.set_ans.resize(r.sets.size());      // (records are fully written by the executor)
    if (r.reduce_ans.size() < r.reduces.size()) r.reduce_ans.resize(r.reduces.size());
    const size_t n_pairs = r.edge_has_target.size();
    if (r.edge_ans.size() < n_pairs) r.edge_ans.resize(n_pairs);
    if (r.proj_ans.size() < r.projs.size()) r.proj_ans.resize(r.projs.size());
    r.path_out.assign(r.paths.size() * (size_t)MAX_PATH, -1);
    r.path_len.assign(r.paths.size(), -1);
    if (stats) {
      stats->set_requests += (long long)r.sets.size(); stats->edge_pairs += (long long)n_pairs;
      stats->projections += (long long)r.projs.size(); stats->paths += (long long)r.paths.size();
    }
    if (stats) stats->gather_ms += now_ms() - t_g0;
    if (ex.submit(l, r, qs)) return -1;
    in_flight[l] = 1;
    return (int)live;
  };
  // resume the queries of lane l with the answers of its round
  HostPool pool(par.threads);
  pool.min_items = (size_t)std::max(1, par.pool_min);
  struct Task { int owner; const SetAns* sa; const EdgeAns* ea; const ProjAns* pa; const int* path; int path_len; };
  std::vector<Task> tasks;
  auto deliver = [&](int l) {
    const double t_d0 = now_ms();
    Round& r = rounds_[l];
    tasks.clear();
    for (size_t k = 0; k < r.sets.size(); ++k) tasks.push_back(Task{r.set_owner[k], &r.set_ans[k], nullptr, nullptr, nullptr, 0});
    for (size_t k = 0; k < r.edges.size(); ++k)
      tasks.push_back(Task{r.edge_owner[k], nullptr, r.edge_ans.data() + r.edges[k].first_pair, nullptr, nullptr, 0});
    size_t po = 0;
    for (size_t k = 0; k < r.proj_owner.size(); ++k) {
      tasks.push_back(Task{r.proj_owner[k], nullptr, nullptr, r.proj_ans.data() + po, nullptr, 0});
      po += (size_t)r.proj_count[k];
    }
    for (size_t k = 0; k < r.paths.size(); ++k)
      tasks.push_back(Task{r.path_owner[k], nullptr, nullptr, nullptr, r.path_out.data() + k * (size_t)MAX_PATH, r.path_len[k]});
    for (size_t k = 0; k < r.reduces.size(); ++k)
      tasks.push_back(Task{r.reduce_owner[k], &r.reduce_ans[k], nullptr, nullptr, nullptr, 0});
    // one task per live query of the lane: the state machines are independent of each other
    const std::function<void(size_t)> fn = [&](size_t k) {
      const Task& t = tasks[k];
      qs[(size_t)t.owner].resume(t.sa, t.ea, t.pa, t.path, t.path_len);
    };
    pool.parallel_for(tasks.size(), fn);
    for (size_t i = (size_t)l; i < qs.size(); i += (size_t)L)
      if (!qs[i].finished) qs[i].rounds = n_rounds[l];
    if (stats) stats->resume_ms += now_ms() - t_d0;
  };

  for (int l = 0; l < L; ++l)
    if (launch(l) < 0) return 9;
  for (;;) {
    bool any = false;
    for (int l = 0; l < L; ++l) {
      if (!in_flight[l]) continue;
      any = true;
      if (ex.collect(l, rounds_[l])) return 9;
      in_flight[l] = 0;
      deliver(l);
      if (launch(l) < 0) return 9;           // (the other lanes' rounds run on the device meanwhile)
    }
    if (!any) break;
  }
  if (stats) stats->rounds = *std::max_element(n_rounds.begin(), n_rounds.end());
  return 0;
}

}  // namespace bpplan

// (the flat C views of a batch, bp_plan_in / bp_plan_out, are declared in include/bpgeo.h)

namespace bpplan {

// The replanning inputs of a batch (bp_plan_in, ABI 4): "" when they are well-formed, else what is wrong.
inline std::string check_replan_inputs(const bp_plan_in& in) {
  char buf[160];
  const int Q = in.Q;
  bool any_replan = false;
  for (int q = 0; in.replanning && q < Q; ++q) any_replan = any_replan || in.replanning[q] != 0;
  if (any_replan && !in.horizon_off) return "replanning queries without horizon_off";
  if (in.horizon_off) {
    if (in.horizon_off[0] != 0) return "horizon_off[0] is not 0";
    for (int q = 0; q < Q; ++q)
      if (in.horizon_off[q + 1] < in.horizon_off[q]) {
        snprintf(buf, sizeof(buf), "horizon_off decreases at query %d", q);
        return buf;
      }
    if (in.horizon_off[Q] > 0 && !in.p_horizon) return "horizon points without p_horizon";
  }
  if (in.prev_off) {
    if (in.prev_off[0] != 0) return "prev_off[0] is not 0";
    for (int q = 0; q < Q; ++q) {
      const int n = in.prev_off[q + 1] - in.prev_off[q];
      if (n < 0) {
        snprintf(buf, sizeof(buf), "prev_off decreases at query %d", q);
        return buf;
      }
      if (n > MAX_PREV_SETS) {
        snprintf(buf, sizeof(buf), "query %d has %d previous sets (at most %d)", q, n, MAX_PREV_SETS);
        return buf;
      }
    }
    const int n_prev = in.prev_off[Q];
    if (n_prev > 0 && (!in.prev_row_off || !in.prev_rows)) return "previous sets without prev_row_off / prev_rows";
    if (n_prev > 0 && in.prev_row_off[0] != 0) return "prev_row_off[0] is not 0";
    for (int s = 0; s < n_prev; ++s) {
      const int m = in.prev_row_off[s + 1] - in.prev_row_off[s];
      if (m < 1 || m > SET_ROWS) {
        snprintf(buf, sizeof(buf), "previous set %d has %d rows (1 .. %d)", s, m, SET_ROWS);
        return buf;
      }
    }
  }
  return "";
}

// query_scene [Q] (or NULL: query q plans in scene q): query q's obstacles are scene query_scene[q]'s, i.e.
// in.box_off has one entry per scene + 1 and the boxes / obs_rows of every scene appear once
inline void load_queries(const bp_plan_in& in, Params& par, std::vector<Query>& qs, const int* query_scene = nullptr) {
  par.obs_size_increase = in.inflate;
  for (int k = 0; k < 3; ++k) { par.ws_min[k] = in.ws_min[k]; par.ws_max[k] = in.ws_max[k]; }
  if (in.sample_chunk > 0) par.sample_chunk = in.sample_chunk;
  if (in.max_rounds > 0) par.max_rounds = in.max_rounds;
  {
    // host threads for the resume loop: BPGEO_PLAN_THREADS, else up to four of the cores this process may use
    int th = 0;
    if (const char* ev = getenv("BPGEO_PLAN_THREADS")) th = atoi(ev);
    if (th <= 0) th = (int)std::min(4u, std::max(1u, std::thread::hardware_concurrency()));
    par.threads = std::min(th, 16);
    if (const char* ev = getenv("BPGEO_PLAN_POOL_MIN")) par.pool_min = std::max(1, atoi(ev));
  }
  qs.clear();
  qs.resize((size_t)in.Q);
  for (int q = 0; q < in.Q; ++q) {
    QueryInput qi;
    const int s = query_scene ? query_scene[q] : q;
    qi.boxes = in.obs_rows ? nullptr : in.boxes + 6 * (size_t)in.box_off[s];
    qi.obs_rows = in.obs_rows ? in.obs_rows + (size_t)OBS_ROWS * 4 * in.box_off[s] : nullptr;
    qi.n_obs = in.box_off[s + 1] - in.box_off[s];
    for (int k = 0; k < 3; ++k) {
      qi.start[k] = in.starts[3 * q + k]; qi.end[k] = in.ends[3 * q + k];
      qi.l_ee[k] = in.l_ee[3 * q + k]; qi.l_ee_end[k] = in.l_ee_end[3 * q + k];
    }
    std::memcpy(qi.ee_samples, in.ee_samples + (size_t)q * FIT_SAMPLES * 3, sizeof(qi.ee_samples));
    for (int k = 0; k < 4; ++k) qi.rng[k] = in.rng[4 * q + k];
    qi.has_first_sample = in.has_first ? in.has_first[q] : 0;
    for (int k = 0; k < 3; ++k) qi.first_sample[k] = (in.first_sample && qi.has_first_sample) ? in.first_sample[3 * q + k] : 0.0;
    qi.replanning = in.replanning ? in.replanning[q] : 0;
    qi.new_obs = in.new_obs ? in.new_obs[q] : 0;
    qi.n_horizon = in.horizon_off ? in.horizon_off[q + 1] - in.horizon_off[q] : 0;
    qi.p_horizon = in.horizon_off && in.p_horizon ? in.p_horizon + 3 * (size_t)in.horizon_off[q] : nullptr;
    qi.n_prev = in.prev_off ? in.prev_off[q + 1] - in.prev_off[q] : 0;
    qi.prev_row_off = in.prev_off && in.prev_row_off ? in.prev_row_off + in.prev_off[q] : nullptr;
    qi.prev_rows = in.prev_rows;
    qs[(size_t)q].init(q, &par, qi);
    qs[(size_t)q].scene = s;
  }
}

inline void store_results(const std::vector<Query>& qs, const RunStats& st, const int* finish_round, const double* finish_ms,
                          bp_plan_out& out) {
  for (size_t q = 0; q < qs.size(); ++q) {
    const Query& Qy = qs[q];
    out.err_kind[q] = Qy.err_kind;
    std::snprintf(out.err_msg + 160 * q, 160, "%s", Qy.err_msg.c_str());
    const int pl = Qy.err_kind ? 0 : (int)std::min<size_t>(Qy.path.size(), MAX_PATH);
    out.path_len[q] = pl;
    for (int k = 0; k < pl; ++k) out.path[MAX_PATH * q + k] = Qy.path[k];
    const int ni = Qy.err_kind ? 0 : (int)std::min<size_t>(Qy.set_ids.size(), MAX_PATH);
    out.n_ids[q] = ni;
    for (int k = 0; k < ni; ++k) out.set_ids[MAX_PATH * q + k] = Qy.set_ids[k];
    const int nv = Qy.err_kind ? 0 : (int)std::min<size_t>(Qy.p_via.size() / 3, MAX_PATH + 2);
    out.n_via[q] = nv;
    for (int k = 0; k < 3 * nv; ++k) out.p_via[(MAX_PATH + 2) * 3 * q + k] = Qy.p_via[k];
    if (out.rng_out) Qy.rng.get((uint64_t*)out.rng_out + 4 * q);
    out.n_nodes[q] = (int)Qy.nodes.size();
    out.n_inter[q] = (int)Qy.inter.size();
    int ne = 0;
    for (const Inter& it : Qy.inter) ne += (int)it.adj.size();
    out.n_edges[q] = ne / 2;
    out.finish_round[q] = finish_round[q];
    if (out.p_horizon_max)
      for (int k = 0; k < 3; ++k) out.p_horizon_max[3 * q + k] = Qy.p_horizon_max[k];
    if (out.finish_ms) out.finish_ms[q] = finish_ms ? std::max(finish_ms[q], 0.0) : 0.0;
    if (out.node_A && out.node_b && out.node_m) {
      for (size_t n = 0; n < (size_t)MAX_NODES; ++n) {
        const size_t slot = q * MAX_NODES + n;
        if (n < Qy.nodes.size()) {
          out.node_m[slot] = Qy.nodes[n].m;
          std::memcpy(out.node_A + slot * NODE_ROWS * 3, Qy.nodes[n].A, sizeof(double) * NODE_ROWS * 3);
          std::memcpy(out.node_b + slot * NODE_ROWS, Qy.nodes[n].b, sizeof(double) * NODE_ROWS);
        } else {
          out.node_m[slot] = 0;
        }
      }
    }
  }
  if (out.stats) {
    out.stats[0] = st.rounds; out.stats[1] = st.set_requests; out.stats[2] = st.edge_pairs;
    out.stats[3] = st.projections; out.stats[4] = st.paths;
  }
}

}  // namespace bpplan
