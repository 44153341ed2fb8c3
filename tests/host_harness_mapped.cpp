// tests/host_harness_mapped.cpp -- TEST-ONLY: the host harness (host_harness.cpp, included whole) plus the native
// lock-step driver as bp_plan_run runs it on a plan from bp_plan_create_mapped, with every request answered by the
// harness' callbacks (tests/test_shared_scenes.py builds it into its own library).
#include "host_harness.cpp"

extern "C" {

// query q's obstacles are scene query_scene[q]'s: in->box_off has one entry per scene + 1 and in->boxes / obs_rows
// hold every scene once.  Returns 3 (and err_msg[0] = the reason) when check_replan_inputs rejects the replanning
// inputs, before any callback runs, as hh_plan_batch does.
int hh_plan_batch_mapped(const bp_plan_in* in, const int* query_scene, bp_plan_out* out, hh_cb_set cb_set,
                         hh_cb_edges cb_edges, hh_cb_project cb_project, hh_cb_path cb_path, hh_cb_reduce cb_reduce,
                         int lanes) {
  const std::string bad = bpplan::check_replan_inputs(*in);
  if (!bad.empty()) {
    std::snprintf(out->err_msg, 160, "%s", bad.c_str());
    return 3;
  }
  bpplan::Params par;
  std::vector<bpplan::Query> qs;
  bpplan::load_queries(*in, par, qs, query_scene);
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

}  // extern "C"
