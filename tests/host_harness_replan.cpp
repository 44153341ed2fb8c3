// tests/host_harness_replan.cpp -- TEST-ONLY host build of the native lock-step planner driver (csrc/bp_planner.h)
// with every request kind answered by callbacks, the reduce request of the replanning start fallback included: the
// CPU test plugs the oracle in and compares with the Python planner (tests/test_planner_replanning.py).  It is NOT
// part of the product: boundplanner_b200/ never loads it and libbpgeo.so has no CPU path.
#include "../boundplanner_b200/csrc/bp_planner.h"

extern "C" {

typedef int (*hr_cb_set)(int qid, const bpplan::SetReq* req, int n_nodes, const bpplan::Node* nodes, bpplan::SetAns* out);
typedef int (*hr_cb_edges)(int qid, int id_new, int n_nodes, const bpplan::Node* nodes, const int* has_target,
                           const double* xd, bpplan::EdgeAns* out);
typedef int (*hr_cb_project)(int qid, int id0, int id1, const double* xd, int n_nodes, const bpplan::Node* nodes,
                             bpplan::ProjAns* out);
typedef int (*hr_cb_path)(int qid, int n_nodes, const int* edge_off, const int* edge_dst, const double* edge_w,
                          int* path_out, int* path_len);
// reduce_ineqs of a given set (the start fallback's previous end set): fills out->m_red, Ar, br
typedef int (*hr_cb_reduce)(int qid, const bpplan::ReduceReq* req, bpplan::SetAns* out);

}  // extern "C"

struct HrCallbackExecutor : bpplan::Executor {
  hr_cb_set cb_set; hr_cb_edges cb_edges; hr_cb_project cb_project; hr_cb_path cb_path; hr_cb_reduce cb_reduce;
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

extern "C" {

// the driver over a bp_plan_in with replanning inputs: returns 3 (and err_msg[0] = the reason) when
// check_replan_inputs rejects them, before any callback runs
int hr_plan_batch(const bp_plan_in* in, bp_plan_out* out, hr_cb_set cb_set, hr_cb_edges cb_edges,
                  hr_cb_project cb_project, hr_cb_path cb_path, hr_cb_reduce cb_reduce, int lanes) {
  const std::string bad = bpplan::check_replan_inputs(*in);
  if (!bad.empty()) {
    std::snprintf(out->err_msg, 160, "%s", bad.c_str());
    return 3;
  }
  bpplan::Params par;
  std::vector<bpplan::Query> qs;
  bpplan::load_queries(*in, par, qs);
  HrCallbackExecutor ex;
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

// sizes of the records the Python side mirrors with ctypes
int hr_sizeof(int what) {
  switch (what) {
    case 0: return (int)sizeof(bpplan::SetReq);
    case 1: return (int)sizeof(bpplan::SetAns);
    case 2: return (int)sizeof(bpplan::Node);
    case 3: return (int)sizeof(bp_plan_in);
    case 4: return (int)sizeof(bp_plan_out);
    case 5: return (int)sizeof(bpplan::ReduceReq);
    default: return -1;
  }
}

}  // extern "C"
