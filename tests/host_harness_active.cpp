// tests/host_harness_active.cpp -- TEST-ONLY: the host harness (host_harness.cpp, included whole) plus the native
// lock-step driver as bp_plan_run_active runs it: only the queries with active[q] != 0 are planned, every request
// answered by the harness' callbacks (tests/test_corridor_hits.py builds it into its own library).
#include "host_harness.cpp"

extern "C" {

// query_scene [Q] or NULL (query q plans in scene q, as hh_plan_batch); active [Q] or NULL (every query).  Returns 3
// (and err_msg[0] = the reason) when check_replan_inputs rejects the replanning inputs, before any callback runs, as
// hh_plan_batch does.
int hh_plan_batch_active(const bp_plan_in* in, const int* query_scene, const int* active, bp_plan_out* out,
                         hh_cb_set cb_set, hh_cb_edges cb_edges, hh_cb_project cb_project, hh_cb_path cb_path,
                         hh_cb_reduce cb_reduce, int lanes) {
  const std::string bad = bpplan::check_replan_inputs(*in);
  if (!bad.empty()) {
    std::snprintf(out->err_msg, 160, "%s", bad.c_str());
    return 3;
  }
  bpplan::Params par;
  std::vector<bpplan::Query> qs;
  bpplan::load_queries(*in, par, qs, query_scene, active);
  HhCallbackExecutor ex;
  ex.cb_set = cb_set; ex.cb_edges = cb_edges; ex.cb_project = cb_project; ex.cb_path = cb_path; ex.cb_reduce = cb_reduce;
  ex.n_lanes = lanes > 0 ? lanes : 1;
  bpplan::RunStats st;
  std::vector<int> fin(qs.size(), -1);
  std::vector<double> fin_ms(qs.size(), -1.0);
  const int rc = bpplan::run_lockstep(qs, ex, par, &st, fin.data(), fin_ms.data(), active);
  if (rc) return rc;
  bpplan::store_results(qs, st, fin.data(), fin_ms.data(), *out, active);
  return 0;
}

}  // extern "C"
