// bp_plan_gpu.cuh -- device side of the native lock-step planner driver (bp_plan_*; host core: bp_planner.h).
// Included at the end of bpgeo.cu: it launches that file's kernels directly.
//
// One lock-step round = the pending requests of all live queries, answered by one chain of kernels on `stream`:
//   H2D of the round's input arena (one copy)
//   new graph nodes:  k_set_aabb (their boxes) -> k_plan_commit (rows, box, ellipsoid into the per-query tables)
//   set requests:     k_sample_filter (K11, sampling requests) -> k_plan_gather_seeds -> K5 (optimised / single
//                     pass groups) | K2+K3' (segment sets) | k_plan_scatter_rows (given sets to reduce: the previous
//                     end set of the start fallback) -> K12 (duplicate distance) -> K8 (reduce_ineqs, all groups)
//   add_edges:        k_pair_list (K6) on the node tables -> k_fit_check (K9) per end-effector group
//   projections:      k_project (K10) on the node tables
//   shortest paths:   k_shortest_path (K13)
//   D2H of the round's output arena (one copy), one stream synchronisation.
// The queries' graph nodes stay resident in device tables of MAX_NODES slots per query (reduced rows, box,
// ellipsoid); edge / projection requests refer to them by slot, so only indices and points travel.
#pragma once
#include <chrono>

#include "bp_planner.h"

__global__ void __launch_bounds__(128) k_plan_commit(const int* __restrict__ slots, const double* __restrict__ A,
                                                     const double* __restrict__ b, const int* __restrict__ m,
                                                     const double* __restrict__ q, const double* __restrict__ p,
                                                     const double* __restrict__ aabb, double* tabA, double* tabb,
                                                     int* tabm, double* tabq, double* tabp, double* tabaabb) {
  constexpr int R = bpplan::NODE_ROWS;
  const int i = blockIdx.x, t = threadIdx.x;
  const size_t s = (size_t)slots[i];
  if (t < R * 3) tabA[s * R * 3 + t] = A[(size_t)i * R * 3 + t];
  if (t < R) tabb[s * R + t] = b[(size_t)i * R + t];
  if (t < 9) tabq[s * 9 + t] = q[(size_t)i * 9 + t];
  if (t < 3) tabp[s * 3 + t] = p[(size_t)i * 3 + t];
  if (t < 6) tabaabb[s * 6 + t] = aabb[(size_t)i * 6 + t];
  if (t == 0) tabm[s] = m[i];
}

// seeds[slot[i]] = the first accepted candidate of sampling request i (candidate 0 when none was accepted: that
// set is built and ignored, as in the Python driver)
__global__ void k_plan_gather_seeds(const double* __restrict__ cand, const int* __restrict__ first,
                                    const int* __restrict__ slot, int C, int n, double* seeds) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int f = first[i] > 0 ? first[i] : 0;
#pragma unroll
  for (int k = 0; k < 3; ++k) seeds[3 * (size_t)slot[i] + k] = cand[((size_t)i * C + f) * 3 + k];
}

// set i of a round's reduce group = rows row_off[i] .. row_off[i+1]-1 of rows [.,4] (a0, a1, a2, b), padded to m_max
// rows with A = 0, b = 10 (what bp_reduce_ineqs takes)
__global__ void __launch_bounds__(64) k_plan_scatter_rows(const int* __restrict__ row_off, const double* __restrict__ rows,
                                                          int m_max, double* A, double* b, int* m) {
  const int i = blockIdx.x;
  const int r0 = row_off[i], n = row_off[i + 1] - r0;
  for (int t = threadIdx.x; t < m_max; t += blockDim.x) {
    const size_t o = (size_t)i * m_max + t;
    const double* src = rows + 4 * (size_t)(r0 + t);
#pragma unroll
    for (int k = 0; k < 3; ++k) A[3 * o + k] = t < n ? src[k] : 0.0;
    b[o] = t < n ? src[3] : 10.0;
  }
  if (threadIdx.x == 0) m[i] = n;
}

// One lock-step lane: its own streams, arenas and build workspace; the node tables are shared (disjoint slots).
struct PlanLane {
  // shared with the other lanes (set by bp_plan_create / bp_plan_run)
  const bp_scene* scene = nullptr;
  int Q = 0;
  double *tabA = nullptr, *tabb = nullptr, *tabq = nullptr, *tabp = nullptr, *tabaabb = nullptr;
  int* tabm = nullptr;
  const std::vector<int>* ee_group_p = nullptr;                  // [Q] end-effector group of every query
  const std::vector<const double*>* ee_samples_p = nullptr;      // the groups' 20 offsets (host)
  double ws_min[3], ws_max[3];
  bool trace = false;
  // per lane
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;           // add_edges / projection / shortest-path chain, concurrent with the set builds
  bool own_stream = false;
  cudaEvent_t ev_in = nullptr, ev_side = nullptr;
  void* work = nullptr;
  size_t work_bytes = 0;
  // arenas (pinned host mirror + device), bump-allocated every round
  char *h_in = nullptr, *d_in = nullptr, *h_out = nullptr, *d_out = nullptr;
  size_t in_cap = 0, out_cap = 0, in_used = 0, out_used = 0;
  // nodes committed since the last round
  std::vector<int> new_slots;
  std::vector<bpplan::Node> new_nodes;
  long long chains = 0, wait_us = 0, pack_us = 0, launch_us = 0, unpack_us = 0;
  std::string error;
  // what collect() needs to know about the round submit() laid out
  struct Layout {
    int nS = 0, nR = 0, nE = 0, nProj = 0, nG = 0, nSmp = 0, nPairs = 0, nNew = 0;
    int n_grp[3] = {0, 0, 0};
    std::vector<int> order, smp_of, e_off;
    size_t o_A, o_b, o_m, o_q, o_p, o_st, o_peak, o_coll, o_Ar, o_br, o_mr, o_dv, o_first, o_res, o_x, o_fits, o_fk, o_epx,
        o_epst, o_px, o_pst, o_path, o_plen;
  } lay;

  int fail(const char* what, cudaError_t e = cudaSuccess) {
    error = what;
    if (e != cudaSuccess) { error += ": "; error += cudaGetErrorString(e); }
    return 9;
  }

  int reserve(size_t in_bytes, size_t out_bytes) {
    if (in_bytes > in_cap) {
      if (h_in) cudaFreeHost(h_in);
      if (d_in) cudaFree(d_in);
      in_cap = in_bytes + in_bytes / 2;
      if (cudaMallocHost(&h_in, in_cap) != cudaSuccess || cudaMalloc(&d_in, in_cap) != cudaSuccess) return fail("bp_plan: arena allocation");
    }
    if (out_bytes > out_cap) {
      if (h_out) cudaFreeHost(h_out);
      if (d_out) cudaFree(d_out);
      out_cap = out_bytes + out_bytes / 2;
      if (cudaMallocHost(&h_out, out_cap) != cudaSuccess || cudaMalloc(&d_out, out_cap) != cudaSuccess) return fail("bp_plan: arena allocation");
    }
    return 0;
  }
  static size_t al(size_t x) { return (x + 15) & ~(size_t)15; }
  size_t take_in(size_t bytes) { const size_t o = in_used; in_used += al(bytes); return o; }
  size_t take_out(size_t bytes) { const size_t o = out_used; out_used += al(bytes); return o; }

  void commit_node(int qid, int node_id, const bpplan::Node& n) {
    new_slots.push_back(qid * bpplan::MAX_NODES + node_id);
    new_nodes.push_back(n);
  }

  int submit(bpplan::Round& r, const std::vector<bpplan::Query>& qs) {
    const std::vector<int>& ee_group = *ee_group_p;
    const std::vector<const double*>& ee_group_samples = *ee_samples_p;
    using namespace bpplan;
    const auto t_pack = std::chrono::steady_clock::now();
    constexpr int R = NODE_ROWS, M = SET_ROWS;
    const int S_tab = Q * MAX_NODES;
    // ---- order the set requests: optimised point sets | single-pass point sets | segment sets
    const int nS = (int)r.sets.size();
    std::vector<int> order;
    order.reserve(nS);
    int n_grp[3] = {0, 0, 0};
    for (int g = 0; g < 3; ++g)
      for (int k = 0; k < nS; ++k) {
        const SetReq& s = r.sets[k];
        const int grp = s.kind == SET_LINE ? 2 : (s.optimize ? 0 : 1);
        if (grp == g) { order.push_back(k); ++n_grp[g]; }
        if (g == 0 && s.kind != SET_LINE && !s.fixed_mid) return fail("bp_plan: free-centre point sets are not part of the planner loop");
      }
    const int nP = n_grp[0] + n_grp[1], nL = n_grp[2];
    int nSmp = 0, C = 1;
    for (int k = 0; k < nS; ++k)
      if (r.sets[k].kind == SET_SAMPLE) { ++nSmp; C = std::max(C, r.sets[k].n_cand); }
    // ---- edge pairs, by end-effector group
    const int nE = (int)r.edges.size();
    std::vector<int> e_off(nE, 0);
    std::vector<std::pair<int, int>> grp_range;      // (first pair, count) per group, in ee_group_samples order
    int nPairs = 0;
    for (size_t g = 0; g < ee_group_samples.size(); ++g) {
      const int first = nPairs;
      for (int k = 0; k < nE; ++k)
        if (ee_group[r.edges[k].qid] == (int)g) { e_off[k] = nPairs; nPairs += r.edges[k].n_others; }
      grp_range.emplace_back(first, nPairs - first);
    }
    const int nProj = (int)r.projs.size(), nG = (int)r.paths.size();
    const int nNew = (int)new_slots.size();
    const int nNodesCsr = nG ? r.node_off.back() : 0, nEdgesCsr = (int)r.edge_dst.size();
    // given sets to reduce: a fourth group after the set builds, in the same output slots (K8 reduces them all)
    const int nR = (int)r.reduces.size(), nSet = nS + nR;
    int nRows = 0;
    for (const ReduceReq& rq : r.reduces) nRows += rq.m;

    // ---- arena layout
    in_used = out_used = 0;
    const size_t need_in = 64 * 16 + al(sizeof(int) * nNew) + al(sizeof(double) * nNew * R * 3) + al(sizeof(double) * nNew * R) +
                           al(sizeof(int) * nNew) + al(sizeof(double) * nNew * 9) + al(sizeof(double) * nNew * 3) +
                           2 * al(sizeof(double) * nS * 3) + 3 * al(sizeof(int) * nS) +
                           al(sizeof(double) * (size_t)nSmp * C * 3) + 4 * al(sizeof(int) * nSmp) +
                           al(sizeof(int) * 2 * nPairs) + al(sizeof(int) * nPairs) + al(sizeof(double) * 3 * nPairs) +
                           al(sizeof(int) * 2 * nProj) + al(sizeof(double) * 3 * nProj) +
                           al(sizeof(int) * (nG + 1)) + 2 * al(sizeof(int) * nG) + al(sizeof(int) * (nNodesCsr + 1)) +
                           al(sizeof(int) * nEdgesCsr) + al(sizeof(double) * nEdgesCsr) + al(sizeof(int) * (nR + 1)) +
                           al(sizeof(double) * 4 * nRows);
    const size_t need_out = 64 * 16 + al(sizeof(double) * nNew * 6) + 2 * al(sizeof(double) * nSet * M * 3) +
                            2 * al(sizeof(double) * nSet * M) + al(sizeof(double) * nS * 9) + al(sizeof(double) * nS * 3) +
                            8 * al(sizeof(int) * nSet) + al(sizeof(double) * nS) + al(sizeof(double) * nS * 3) + al(sizeof(int) * nSmp) +
                            4 * al(sizeof(int) * nPairs) + 2 * al(sizeof(double) * 3 * nPairs) + al(sizeof(double) * 3 * nProj) +
                            al(sizeof(int) * nProj) + al(sizeof(int) * nG * MAX_PATH) + al(sizeof(int) * nG) + al(sizeof(double) * nG);
    if (int rc = reserve(need_in, need_out)) return rc;
#define IN_H(T, off) ((T*)(h_in + (off)))
#define IN_D(T, off) ((T*)(d_in + (off)))
#define OUT_H(T, off) ((T*)(h_out + (off)))
#define OUT_D(T, off) ((T*)(d_out + (off)))
    // new nodes
    const size_t i_slot = take_in(sizeof(int) * nNew), i_nA = take_in(sizeof(double) * nNew * R * 3),
                 i_nb = take_in(sizeof(double) * nNew * R), i_nm = take_in(sizeof(int) * nNew),
                 i_nq = take_in(sizeof(double) * nNew * 9), i_np = take_in(sizeof(double) * nNew * 3);
    for (int i = 0; i < nNew; ++i) {
      IN_H(int, i_slot)[i] = new_slots[i];
      memcpy(IN_H(double, i_nA) + (size_t)i * R * 3, new_nodes[i].A, sizeof(double) * R * 3);
      memcpy(IN_H(double, i_nb) + (size_t)i * R, new_nodes[i].b, sizeof(double) * R);
      IN_H(int, i_nm)[i] = new_nodes[i].m;
      memcpy(IN_H(double, i_nq) + (size_t)i * 9, new_nodes[i].Q, sizeof(double) * 9);
      memcpy(IN_H(double, i_np) + (size_t)i * 3, new_nodes[i].P, sizeof(double) * 3);
    }
    // set requests
    const size_t i_p0 = take_in(sizeof(double) * nS * 3), i_p1 = take_in(sizeof(double) * nS * 3),
                 i_scene = take_in(sizeof(int) * nS), i_nbeg = take_in(sizeof(int) * nS), i_ncnt = take_in(sizeof(int) * nS),
                 i_cand = take_in(sizeof(double) * (size_t)nSmp * C * 3), i_sslot = take_in(sizeof(int) * nSmp),
                 i_sscene = take_in(sizeof(int) * nSmp), i_sbeg = take_in(sizeof(int) * nSmp), i_scnt = take_in(sizeof(int) * nSmp);
    std::vector<int> smp_of(nS, -1);
    {
      int js = 0;
      for (int j = 0; j < nS; ++j) {
        const SetReq& s = r.sets[order[j]];
        const Query& q = qs[r.set_owner[order[j]]];
        for (int k = 0; k < 3; ++k) { IN_H(double, i_p0)[3 * j + k] = s.p0[k]; IN_H(double, i_p1)[3 * j + k] = s.p1[k]; }
        IN_H(int, i_scene)[j] = q.scene;                  // (the node tables stay per query)
        IN_H(int, i_nbeg)[j] = s.qid * MAX_NODES;
        IN_H(int, i_ncnt)[j] = s.with_dv ? (int)q.nodes.size() : 0;
        if (s.kind == SET_SAMPLE) {
          double* c = IN_H(double, i_cand) + (size_t)js * C * 3;
          memcpy(c, s.cand, sizeof(double) * 3 * s.n_cand);
          for (int e = s.n_cand; e < C; ++e) memcpy(c + 3 * e, s.cand, sizeof(double) * 3);   // padding never wins
          IN_H(int, i_sslot)[js] = j;
          IN_H(int, i_sscene)[js] = q.scene;
          IN_H(int, i_sbeg)[js] = s.qid * MAX_NODES;
          IN_H(int, i_scnt)[js] = (int)q.nodes.size();
          smp_of[j] = js++;
        }
      }
    }
    // edges / projections / paths
    const size_t i_pairs = take_in(sizeof(int) * 2 * nPairs), i_ehas = take_in(sizeof(int) * nPairs),
                 i_exd = take_in(sizeof(double) * 3 * nPairs), i_ppairs = take_in(sizeof(int) * 2 * nProj),
                 i_xd = take_in(sizeof(double) * 3 * nProj);
    for (int k = 0; k < nE; ++k) {
      const EdgeReq& e = r.edges[k];
      int* pp = IN_H(int, i_pairs) + 2 * (size_t)e_off[k];
      for (int v = 0; v < e.n_others; ++v) { pp[2 * v] = e.qid * MAX_NODES + v; pp[2 * v + 1] = e.qid * MAX_NODES + e.id_new; }
      // the point every hit of this request is projected from, when it is known already (see Query::spec_target)
      memcpy(IN_H(int, i_ehas) + e_off[k], r.edge_has_target.data() + e.first_pair, sizeof(int) * e.n_others);
      memcpy(IN_H(double, i_exd) + 3 * (size_t)e_off[k], r.edge_xd.data() + 3 * (size_t)e.first_pair, sizeof(double) * 3 * e.n_others);
    }
    for (int k = 0; k < nProj; ++k) {
      const ProjReq& p = r.projs[k];
      IN_H(int, i_ppairs)[2 * k] = p.qid * MAX_NODES + p.id0;
      IN_H(int, i_ppairs)[2 * k + 1] = p.qid * MAX_NODES + p.id1;
      for (int c = 0; c < 3; ++c) IN_H(double, i_xd)[3 * k + c] = p.xd[c];
    }
    const size_t i_noff = take_in(sizeof(int) * (nG + 1)), i_src = take_in(sizeof(int) * nG), i_dst = take_in(sizeof(int) * nG),
                 i_eoff = take_in(sizeof(int) * (nNodesCsr + 1)), i_edst = take_in(sizeof(int) * nEdgesCsr),
                 i_ew = take_in(sizeof(double) * nEdgesCsr);
    if (nG) {
      memcpy(IN_H(int, i_noff), r.node_off.data(), sizeof(int) * (nG + 1));
      memcpy(IN_H(int, i_eoff), r.edge_off.data(), sizeof(int) * (nNodesCsr + 1));
      if (nEdgesCsr) {
        memcpy(IN_H(int, i_edst), r.edge_dst.data(), sizeof(int) * nEdgesCsr);
        memcpy(IN_H(double, i_ew), r.edge_w.data(), sizeof(double) * nEdgesCsr);
      }
      for (int g = 0; g < nG; ++g) { IN_H(int, i_src)[g] = 0; IN_H(int, i_dst)[g] = 1; }
    }
    const size_t i_roff = take_in(sizeof(int) * (nR + 1)), i_rrows = take_in(sizeof(double) * 4 * nRows);
    if (nR) {
      IN_H(int, i_roff)[0] = 0;
      for (int k = 0; k < nR; ++k) {
        const ReduceReq& rq = r.reduces[k];
        memcpy(IN_H(double, i_rrows) + 4 * (size_t)IN_H(int, i_roff)[k], rq.rows, sizeof(double) * 4 * rq.m);
        IN_H(int, i_roff)[k + 1] = IN_H(int, i_roff)[k] + rq.m;
      }
    }
    if (in_used > in_cap) return fail("bp_plan: input arena overflow");
    // outputs
    const size_t o_naabb = take_out(sizeof(double) * nNew * 6);
    const size_t o_A = take_out(sizeof(double) * nSet * M * 3), o_b = take_out(sizeof(double) * nSet * M), o_m = take_out(sizeof(int) * nSet),
                 o_q = take_out(sizeof(double) * nS * 9), o_p = take_out(sizeof(double) * nS * 3), o_st = take_out(sizeof(int) * nS),
                 o_it = take_out(sizeof(int) * nS), o_peak = take_out(sizeof(int) * nS), o_coll = take_out(sizeof(int) * nS),
                 o_Ar = take_out(sizeof(double) * nSet * M * 3), o_br = take_out(sizeof(double) * nSet * M), o_mr = take_out(sizeof(int) * nSet),
                 o_rst = take_out(sizeof(int) * nSet), o_dv = take_out(sizeof(double) * nS), o_arg = take_out(sizeof(int) * nS),
                 o_seed = take_out(sizeof(double) * nS * 3), o_first = take_out(sizeof(int) * nSmp);
    const size_t o_res = take_out(sizeof(int) * nPairs), o_x = take_out(sizeof(double) * 3 * nPairs),
                 o_fits = take_out(sizeof(int) * nPairs), o_fk = take_out(sizeof(int) * nPairs),
                 o_epx = take_out(sizeof(double) * 3 * nPairs), o_epst = take_out(sizeof(int) * nPairs),
                 o_px = take_out(sizeof(double) * 3 * nProj), o_pst = take_out(sizeof(int) * nProj),
                 o_path = take_out(sizeof(int) * nG * MAX_PATH), o_plen = take_out(sizeof(int) * nG), o_cost = take_out(sizeof(double) * nG);
    if (out_used > out_cap) return fail("bp_plan: output arena overflow");

    // ---- the kernel chain
    const auto t_launch = std::chrono::steady_clock::now();
    pack_us += std::chrono::duration_cast<std::chrono::microseconds>(t_launch - t_pack).count();
    cudaError_t e = cudaSuccess;
    if (in_used) e = cudaMemcpyAsync(d_in, h_in, in_used, cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return fail("bp_plan: H2D", e);
    if (nNew) {
      k_set_aabb<<<nNew, 128, 0, stream>>>(IN_D(double, i_nA), IN_D(double, i_nb), IN_D(int, i_nm), nNew, R, OUT_D(double, o_naabb));
      k_plan_commit<<<nNew, 128, 0, stream>>>(IN_D(int, i_slot), IN_D(double, i_nA), IN_D(double, i_nb), IN_D(int, i_nm),
                                               IN_D(double, i_nq), IN_D(double, i_np), OUT_D(double, o_naabb), tabA, tabb, tabm,
                                               tabq, tabp, tabaabb);
      new_slots.clear();
      new_nodes.clear();
    }
    // the requests of a round belong to different queries: the set builds (main stream) and the add_edges /
    // projection / shortest-path chain (side stream) run concurrently between the two copies
    const bool fork = nSet && (nPairs || nProj || nG);
    cudaStream_t st2 = fork ? side : stream;
    if (fork) {
      e = cudaEventRecord(ev_in, stream);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(side, ev_in, 0);
      if (e != cudaSuccess) return fail("bp_plan: fork", e);
    }
    if (nS) {
      // the seeds of the point groups: given points are copied, sampled ones gathered from the candidates
      e = cudaMemcpyAsync(OUT_D(double, o_seed), IN_D(double, i_p0), sizeof(double) * 3 * nS, cudaMemcpyDeviceToDevice, stream);
      if (e != cudaSuccess) return fail("bp_plan: seed copy", e);
      if (nSmp) {
        if (bp_sample_filter_tables(scene, IN_D(int, i_sscene), IN_D(double, i_cand), nSmp, C, tabA, tabb, tabm, R,
                                    IN_D(int, i_sbeg), IN_D(int, i_scnt), OUT_D(int, o_first), stream))
          return fail(bp_last_error_string());
        k_plan_gather_seeds<<<(nSmp + 127) / 128, 128, 0, stream>>>(IN_D(double, i_cand), OUT_D(int, o_first), IN_D(int, i_sslot), C,
                                                                    nSmp, OUT_D(double, o_seed));
      }
      int o = 0;
      for (int g = 0; g < 2; ++g) {
        const int n = n_grp[g];
        if (n && bp_build_sets_point_ms(scene, IN_D(int, i_scene) + o, OUT_D(double, o_seed) + 3 * o, n, ws_min, ws_max, 1, g == 0, 5, M,
                                        OUT_D(double, o_A) + (size_t)o * M * 3, OUT_D(double, o_b) + (size_t)o * M, OUT_D(int, o_m) + o,
                                        OUT_D(double, o_q) + (size_t)o * 9, OUT_D(double, o_p) + (size_t)o * 3, OUT_D(int, o_st) + o,
                                        OUT_D(int, o_it) + o, OUT_D(int, o_peak) + o, REF_MAX_ROWS, work, work_bytes, stream))
          return fail(bp_last_error_string());
        o += n;
      }
      if (nL && bp_build_sets_line_ms(scene, IN_D(int, i_scene) + o, IN_D(double, i_p0) + 3 * o, IN_D(double, i_p1) + 3 * o, nL, ws_min,
                                      ws_max, 0, 0.3, 1, M, OUT_D(double, o_A) + (size_t)o * M * 3, OUT_D(double, o_b) + (size_t)o * M,
                                      OUT_D(int, o_m) + o, OUT_D(double, o_q) + (size_t)o * 9, OUT_D(double, o_p) + (size_t)o * 3,
                                      OUT_D(int, o_coll) + o, OUT_D(int, o_st) + o, work, work_bytes, stream))
        return fail(bp_last_error_string());
      if (nP && bp_dedupe_distance_tables(OUT_D(double, o_q), OUT_D(double, o_p), nP, tabq, tabp, IN_D(int, i_nbeg), IN_D(int, i_ncnt),
                                          OUT_D(double, o_dv), OUT_D(int, o_arg), stream))
        return fail(bp_last_error_string());
    }
    if (nR)
      k_plan_scatter_rows<<<nR, 64, 0, stream>>>(IN_D(int, i_roff), IN_D(double, i_rrows), M, OUT_D(double, o_A) + (size_t)nS * M * 3,
                                                 OUT_D(double, o_b) + (size_t)nS * M, OUT_D(int, o_m) + nS);
    if (nSet && bp_reduce_ineqs(OUT_D(double, o_A), OUT_D(double, o_b), OUT_D(int, o_m), nSet, M, OUT_D(double, o_Ar), OUT_D(double, o_br),
                                OUT_D(int, o_mr), nullptr, OUT_D(int, o_rst), stream))
      return fail(bp_last_error_string());
    if (nPairs) {
      k_pair_list<<<(nPairs + 7) / 8, 256, 0, st2>>>(tabA, tabb, tabm, R, 0.01, tabaabb, (const int2*)IN_D(int, i_pairs), nPairs,
                                                        OUT_D(int, o_res), OUT_D(double, o_x));
      for (size_t g = 0; g < grp_range.size(); ++g) {
        const int f = grp_range[g].first, n = grp_range[g].second;
        if (n && bp_check_fit(tabA, tabb, tabm, S_tab, R, IN_D(int, i_pairs) + 2 * (size_t)f, n, OUT_D(double, o_x) + 3 * (size_t)f,
                              OUT_D(int, o_res) + f, ee_group_samples[g], FIT_SAMPLES, 0.001, OUT_D(int, o_fits) + f,
                              OUT_D(int, o_fk) + f, st2))
          return fail(bp_last_error_string());
      }
    }
    if (nPairs)       // the hits' projections from their known targets, gated by the intersection result (K10)
      k_project<<<(nPairs + 7) / 8, 256, 0, st2>>>(tabA, tabb, tabm, R, (const int2*)IN_D(int, i_pairs), nPairs, IN_D(double, i_exd),
                                                   OUT_D(double, o_epx), OUT_D(int, o_epst), OUT_D(int, o_res), IN_D(int, i_ehas));
    if (nProj && bp_project_points(tabA, tabb, tabm, S_tab, R, IN_D(int, i_ppairs), nProj, IN_D(double, i_xd), OUT_D(double, o_px),
                                   OUT_D(int, o_pst), st2))
      return fail(bp_last_error_string());
    if (nG && bp_shortest_paths(IN_D(int, i_noff), IN_D(int, i_eoff), IN_D(int, i_edst), IN_D(double, i_ew), IN_D(int, i_src),
                                IN_D(int, i_dst), nG, MAX_PATH, OUT_D(int, o_path), OUT_D(int, o_plen), OUT_D(double, o_cost), st2))
      return fail(bp_last_error_string());
    if (fork) {
      e = cudaEventRecord(ev_side, side);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, ev_side, 0);
      if (e != cudaSuccess) return fail("bp_plan: join", e);
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail("bp_plan: kernel launch", e);
    if (out_used) e = cudaMemcpyAsync(h_out, d_out, out_used, cudaMemcpyDeviceToHost, stream);
    if (e != cudaSuccess) return fail("bp_plan: D2H", e);
    launch_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t_launch).count();
    // what collect() needs
    lay.nS = nS; lay.nR = nR; lay.nE = nE; lay.nProj = nProj; lay.nG = nG; lay.nSmp = nSmp; lay.nPairs = nPairs; lay.nNew = nNew;
    lay.n_grp[0] = n_grp[0]; lay.n_grp[1] = n_grp[1]; lay.n_grp[2] = n_grp[2];
    lay.order.swap(order); lay.smp_of.swap(smp_of); lay.e_off.swap(e_off);
    lay.o_A = o_A; lay.o_b = o_b; lay.o_m = o_m; lay.o_q = o_q; lay.o_p = o_p; lay.o_st = o_st; lay.o_peak = o_peak;
    lay.o_coll = o_coll; lay.o_Ar = o_Ar; lay.o_br = o_br; lay.o_mr = o_mr; lay.o_dv = o_dv; lay.o_first = o_first;
    lay.o_res = o_res; lay.o_x = o_x; lay.o_fits = o_fits; lay.o_fk = o_fk; lay.o_epx = o_epx; lay.o_epst = o_epst;
    lay.o_px = o_px; lay.o_pst = o_pst; lay.o_path = o_path; lay.o_plen = o_plen;
#undef IN_H
#undef IN_D
#undef OUT_H
#undef OUT_D
    return 0;
  }

  int collect(bpplan::Round& r) {
    using namespace bpplan;
    constexpr int M = SET_ROWS;
#define OUT_H(T, off) ((T*)(h_out + (off)))
    const int nS = lay.nS, nE = lay.nE, nProj = lay.nProj, nG = lay.nG;
    const std::vector<int>&order = lay.order, &smp_of = lay.smp_of, &e_off = lay.e_off;
    const size_t o_A = lay.o_A, o_b = lay.o_b, o_m = lay.o_m, o_q = lay.o_q, o_p = lay.o_p, o_st = lay.o_st, o_peak = lay.o_peak,
                 o_coll = lay.o_coll, o_Ar = lay.o_Ar, o_br = lay.o_br, o_mr = lay.o_mr, o_dv = lay.o_dv, o_first = lay.o_first,
                 o_res = lay.o_res, o_x = lay.o_x, o_fits = lay.o_fits, o_fk = lay.o_fk, o_epx = lay.o_epx, o_epst = lay.o_epst,
                 o_px = lay.o_px, o_pst = lay.o_pst, o_path = lay.o_path, o_plen = lay.o_plen;
    const auto t0 = std::chrono::steady_clock::now();
    cudaError_t e = cudaStreamSynchronize(stream);
    const auto t_unpack = std::chrono::steady_clock::now();
    wait_us += std::chrono::duration_cast<std::chrono::microseconds>(t_unpack - t0).count();
    if (e != cudaSuccess) return fail("bp_plan: round", e);
    ++chains;
    if (trace)
      fprintf(stderr, "bp_plan round %lld: sets %d (opt %d, single %d, line %d; sampled %d) pairs %d proj %d paths %d new %d  wait %lld us\n",
              chains, nS, lay.n_grp[0], lay.n_grp[1], lay.n_grp[2], lay.nSmp, lay.nPairs, nProj, nG, lay.nNew,
              (long long)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count());

    // ---- answers
    for (int j = 0; j < nS; ++j) {
      const int k = order[j];
      const SetReq& s = r.sets[k];
      SetAns& a = r.set_ans[k];
      a.status = OUT_H(int, o_st)[j];
      a.m = OUT_H(int, o_m)[j];
      a.rows_peak = s.kind == SET_LINE ? a.m : OUT_H(int, o_peak)[j];
      a.m_red = OUT_H(int, o_mr)[j];
      a.collision = s.kind == SET_LINE ? OUT_H(int, o_coll)[j] : 0;
      a.first = s.kind == SET_SAMPLE ? OUT_H(int, o_first)[smp_of[j]] : 0;
      a.dv = (s.kind != SET_LINE && s.with_dv) ? OUT_H(double, o_dv)[j] : INFINITY;
      const int m = std::min(std::max(a.m, 0), M), mr = std::min(std::max(a.m_red, 0), M);
      memcpy(a.A, OUT_H(double, o_A) + (size_t)j * M * 3, sizeof(double) * 3 * m);
      memcpy(a.b, OUT_H(double, o_b) + (size_t)j * M, sizeof(double) * m);
      memcpy(a.Ar, OUT_H(double, o_Ar) + (size_t)j * M * 3, sizeof(double) * 3 * mr);
      memcpy(a.br, OUT_H(double, o_br) + (size_t)j * M, sizeof(double) * mr);
      memcpy(a.Q, OUT_H(double, o_q) + (size_t)j * 9, sizeof(double) * 9);
      memcpy(a.P, OUT_H(double, o_p) + (size_t)j * 3, sizeof(double) * 3);
    }
    for (int k = 0; k < lay.nR; ++k) {
      SetAns& a = r.reduce_ans[k];
      const size_t j = (size_t)nS + k;
      a.status = 0;
      a.m = r.reduces[k].m;
      a.m_red = OUT_H(int, o_mr)[j];
      const int mr = std::min(std::max(a.m_red, 0), M);
      memcpy(a.Ar, OUT_H(double, o_Ar) + j * M * 3, sizeof(double) * 3 * mr);
      memcpy(a.br, OUT_H(double, o_br) + j * M, sizeof(double) * mr);
    }
    for (int k = 0; k < nE; ++k) {
      const EdgeReq& er = r.edges[k];
      for (int v = 0; v < er.n_others; ++v) {
        EdgeAns& ea = r.edge_ans[er.first_pair + v];
        const size_t p = (size_t)e_off[k] + v;
        ea.ok = OUT_H(int, o_res)[p] != 0;
        ea.fits = ea.ok && OUT_H(int, o_fits)[p] > 0;
        for (int c = 0; c < 3; ++c) ea.x[c] = OUT_H(double, o_x)[3 * p + c];
        const int fk = OUT_H(int, o_fk)[p];
        ea.omega = fk >= 0 ? (double)fk / (FIT_SAMPLES - 1) : -1.0;
        ea.proj_ok = ea.ok && r.edge_has_target[er.first_pair + v] && OUT_H(int, o_epst)[p] >= 0;
        for (int c = 0; c < 3; ++c) ea.proj[c] = OUT_H(double, o_epx)[3 * p + c];
      }
    }
    for (int k = 0; k < nProj; ++k) {
      for (int c = 0; c < 3; ++c) r.proj_ans[k].x[c] = OUT_H(double, o_px)[3 * k + c];
      r.proj_ans[k].status = OUT_H(int, o_pst)[k];
    }
    for (int g = 0; g < nG; ++g) {
      r.path_len[g] = OUT_H(int, o_plen)[g];
      memcpy(r.path_out.data() + (size_t)g * MAX_PATH, OUT_H(int, o_path) + (size_t)g * MAX_PATH, sizeof(int) * MAX_PATH);
    }
#undef OUT_H
    unpack_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t_unpack).count();
    return 0;
  }

  void release() {
    cudaFree(work);
    if (h_in) cudaFreeHost(h_in);
    if (d_in) cudaFree(d_in);
    if (h_out) cudaFreeHost(h_out);
    if (d_out) cudaFree(d_out);
    if (side) cudaStreamDestroy(side);
    if (own_stream && stream) cudaStreamDestroy(stream);
    if (ev_in) cudaEventDestroy(ev_in);
    if (ev_side) cudaEventDestroy(ev_side);
  }
};

// The executor of bp_plan_run: up to BP_PLAN_LANES independent lock-step groups in flight (query i -> lane i mod L;
// two by default, BPGEO_PLAN_LANES overrides):
// while one lane's kernel chain runs, the host resumes the other lane's queries and packs its next round.
#define BP_PLAN_LANES 4
struct bp_plan : bpplan::Executor {
  const bp_scene* scene = nullptr;
  int Q = 0, L = 1;
  bool mapped = false;                           // created by bp_plan_create_mapped
  std::vector<int> query_scene;                  // [Q] the scene of every query (the identity when not mapped)
  bool polytopes = false;                        // the scene batch holds polytopes (bp_plan_in::obs_rows) or boxes
  double *tabA = nullptr, *tabb = nullptr, *tabq = nullptr, *tabp = nullptr, *tabaabb = nullptr;
  int* tabm = nullptr;
  PlanLane lane[BP_PLAN_LANES];
  std::vector<int> ee_group;                     // [Q]
  std::vector<const double*> ee_group_samples;
  bool trace = getenv("BPGEO_PLAN_TRACE") != nullptr;
  std::string error;

  int lanes() const override { return L; }
  void commit_node(int l, int qid, int node_id, const bpplan::Node& n) override { lane[l].commit_node(qid, node_id, n); }
  int submit(int l, bpplan::Round& r, const std::vector<bpplan::Query>& qs) override {
    const int rc = lane[l].submit(r, qs);
    if (rc) error = lane[l].error;
    return rc;
  }
  int collect(int l, bpplan::Round& r) override {
    const int rc = lane[l].collect(r);
    if (rc) error = lane[l].error;
    return rc;
  }
  void release() {
    cudaFree(tabA); cudaFree(tabb); cudaFree(tabq); cudaFree(tabp); cudaFree(tabaabb); cudaFree(tabm);
    for (int l = 0; l < BP_PLAN_LANES; ++l) lane[l].release();
  }
};

// the per-scene limit of the polytope kernels a round launches (k_iris_fused / k_poly_point, k_poly_line_p,
// k_sample_filter)
static int plan_scene_limits(const bp_scene* sc, const char* fn) {
  if (sc->rows && sc->n > BP_POLY_SCENE_MAX) {
    snprintf(g_err, sizeof(g_err), "%s: polytope scenes hold at most %d obstacles (largest scene: %d)", fn,
             BP_POLY_SCENE_MAX, sc->n);
    return 1;
  }
  return 0;
}

// bp_plan_create / bp_plan_create_mapped once the query -> scene map is known and checked
static int plan_create(const bp_scene* scene_batch, int Q, std::vector<int>&& query_scene, bool mapped, const char* fn,
                       bp_plan** out) {
  // reported here rather than by the first round that builds a set
  if (plan_scene_limits(scene_batch, fn)) return 1;
  bp_plan* pl = new bp_plan();
  pl->scene = scene_batch;
  pl->Q = Q;
  pl->mapped = mapped;
  pl->query_scene = std::move(query_scene);
  pl->polytopes = scene_batch->rows != nullptr;
  // two lanes once there is enough work to split (BPGEO_PLAN_LANES=1 forces plain lock step)
  pl->L = Q >= 32 ? 2 : 1;
  if (const char* ev = getenv("BPGEO_PLAN_LANES")) pl->L = atoi(ev);
  if (pl->L > BP_PLAN_LANES) pl->L = BP_PLAN_LANES;
  if (pl->L < 1 || pl->L > Q) pl->L = 1;
  const size_t n = (size_t)Q * bpplan::MAX_NODES;
  constexpr int R = bpplan::NODE_ROWS;
  cudaError_t e = cudaMalloc(&pl->tabA, sizeof(double) * n * R * 3);
  if (e == cudaSuccess) e = cudaMalloc(&pl->tabb, sizeof(double) * n * R);
  if (e == cudaSuccess) e = cudaMalloc(&pl->tabm, sizeof(int) * n);
  if (e == cudaSuccess) e = cudaMalloc(&pl->tabq, sizeof(double) * n * 9);
  if (e == cudaSuccess) e = cudaMalloc(&pl->tabp, sizeof(double) * n * 3);
  if (e == cudaSuccess) e = cudaMalloc(&pl->tabaabb, sizeof(double) * n * 6);
  for (int l = 0; l < pl->L && e == cudaSuccess; ++l) {
    PlanLane& ln = pl->lane[l];
    ln.scene = scene_batch; ln.Q = Q;
    ln.tabA = pl->tabA; ln.tabb = pl->tabb; ln.tabm = pl->tabm; ln.tabq = pl->tabq; ln.tabp = pl->tabp; ln.tabaabb = pl->tabaabb;
    ln.ee_group_p = &pl->ee_group; ln.ee_samples_p = &pl->ee_group_samples;
    ln.trace = pl->trace;
    ln.work_bytes = bp_build_sets_workspace_bytes(Q);
    e = cudaMalloc(&ln.work, ln.work_bytes);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ln.side, cudaStreamNonBlocking);
    if (e == cudaSuccess && l > 0) {               // (lane 0 runs on the caller's stream)
      e = cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking);
      ln.own_stream = true;
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ln.ev_in, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ln.ev_side, cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaMemset(pl->tabm, 0, sizeof(int) * n);
  if (e == cudaSuccess) e = cudaMemset(pl->tabA, 0, sizeof(double) * n * R * 3);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();        // (the lanes' streams do not order with the memsets)
  if (e != cudaSuccess) {
    pl->release();
    delete pl;
    return bp_fail(fn, e);
  }
  *out = pl;
  return 0;
}

extern "C" {

int bp_plan_create(const bp_scene* scene_batch, int Q, bp_plan** out) {
  if (!scene_batch || Q < 1 || !out) return bp_fail("bp_plan_create: bad arguments");
  if (!scene_batch->seg_off || scene_batch->n_seg != Q) return bp_fail("bp_plan_create: needs a scene batch with one scene per query");
  std::vector<int> ident((size_t)Q);
  for (int q = 0; q < Q; ++q) ident[(size_t)q] = q;
  return plan_create(scene_batch, Q, std::move(ident), false, "bp_plan_create", out);
}

int bp_plan_create_mapped(const bp_scene* scene_batch, int Q, const int* query_scene_host, bp_plan** out) {
  if (!scene_batch || Q < 1 || !query_scene_host || !out) return bp_fail("bp_plan_create_mapped: bad arguments");
  if (!scene_batch->seg_off || scene_batch->n_seg < 1) return bp_fail("bp_plan_create_mapped: needs a scene batch");
  const int n_scenes = scene_batch->n_seg;
  for (int q = 0; q < Q; ++q)
    if (query_scene_host[q] < 0 || query_scene_host[q] >= n_scenes) {
      snprintf(g_err, sizeof(g_err), "bp_plan_create_mapped: query %d maps to scene %d, the batch has %d scenes", q,
               query_scene_host[q], n_scenes);
      return 1;
    }
  return plan_create(scene_batch, Q, std::vector<int>(query_scene_host, query_scene_host + Q), true, "bp_plan_create_mapped",
                     out);
}

}  // extern "C"

// bp_plan_run / bp_plan_run_active: active [Q] or NULL (every query)
static int plan_run(bp_plan* pl, const bp_plan_in* in, const int* active, bp_plan_out* out, void* stream) {
  if (!pl || !in || !out || in->Q != pl->Q || (!in->boxes && !in->obs_rows) || !in->box_off || !in->ws_min || !in->ws_max || !in->starts ||
      !in->ends || !in->l_ee || !in->l_ee_end || !in->ee_samples || !in->rng || !out->err_kind || !out->err_msg ||
      !out->path || !out->path_len || !out->set_ids || !out->n_ids || !out->p_via || !out->n_via || !out->n_nodes ||
      !out->n_inter || !out->n_edges || !out->finish_round)
    return bp_fail("bp_plan_run: bad arguments");
  if (in->sample_chunk > 64) return bp_fail("bp_plan_run: sample_chunk is at most 64");
  // the host pushes `end` out of the obstacles of `in`, the device builds sets around the scene batch: same kind, same
  // obstacle counts (against the scene's host copy of its offsets, which bp_scene_update_*batch keeps current); an
  // update may also have crossed the per-scene limit
  if (pl->polytopes && !in->obs_rows)
    return bp_fail("bp_plan_run: the plan's scene batch holds polytopes, the input has no obs_rows");
  if (!pl->polytopes && in->obs_rows)
    return bp_fail("bp_plan_run: the plan's scene batch holds boxes, the input has obs_rows");
  // (a mapped plan's input holds every scene once: box_off has n_scenes + 1 entries)
  for (int s = 0; s < pl->scene->n_seg; ++s) {
    const int* so = pl->scene->seg_off_host;
    const int n_in = in->box_off[s + 1] - in->box_off[s], n_scene = so[s + 1] - so[s];
    if (n_in != n_scene) {
      if (pl->mapped)
        snprintf(g_err, sizeof(g_err), "bp_plan_run: scene %d has %d obstacles in the input, %d in the plan's scene batch", s,
                 n_in, n_scene);
      else
        snprintf(g_err, sizeof(g_err), "bp_plan_run: query %d has %d obstacles, its scene %d", s, n_in, n_scene);
      return 1;
    }
  }
  if (plan_scene_limits(pl->scene, "bp_plan_run")) return 1;
  const std::string bad = bpplan::check_replan_inputs(*in);
  if (!bad.empty()) return bp_fail(("bp_plan_run: " + bad).c_str());
  bpplan::Params par;
  std::vector<bpplan::Query> qs;
  const auto t_run0 = std::chrono::steady_clock::now();
  bpplan::load_queries(*in, par, qs, pl->query_scene.data(), active);
  const auto t_run1 = std::chrono::steady_clock::now();
  // the work queued on the caller's stream so far precedes the run on every lane
  BP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  pl->ee_group.assign((size_t)pl->Q, 0);
  pl->ee_group_samples.clear();
  for (int q = 0; q < pl->Q; ++q) {
    const double* s = in->ee_samples + (size_t)q * bpplan::FIT_SAMPLES * 3;
    size_t g = 0;
    for (; g < pl->ee_group_samples.size(); ++g)
      if (memcmp(pl->ee_group_samples[g], s, sizeof(double) * bpplan::FIT_SAMPLES * 3) == 0) break;
    if (g == pl->ee_group_samples.size()) pl->ee_group_samples.push_back(s);
    pl->ee_group[(size_t)q] = (int)g;
  }
  for (int l = 0; l < pl->L; ++l) {
    PlanLane& ln = pl->lane[l];
    if (l == 0) ln.stream = (cudaStream_t)stream;
    for (int k = 0; k < 3; ++k) { ln.ws_min[k] = in->ws_min[k]; ln.ws_max[k] = in->ws_max[k]; }
    ln.new_slots.clear();
    ln.new_nodes.clear();
    ln.chains = ln.wait_us = ln.pack_us = ln.launch_us = ln.unpack_us = 0;
  }
  bpplan::RunStats st;
  std::vector<int> fin(qs.size(), -1);
  std::vector<double> fin_ms(qs.size(), -1.0);
  const int rc = bpplan::run_lockstep(qs, *pl, par, &st, fin.data(), fin_ms.data(), active);
  if (rc) {
    for (int l = 0; l < pl->L; ++l) cudaStreamSynchronize(pl->lane[l].stream);       // nothing of the run stays in flight
    return bp_fail(pl->error.empty() ? "bp_plan_run: executor failed" : pl->error.c_str());
  }
  const auto t_run2 = std::chrono::steady_clock::now();
  bpplan::store_results(qs, st, fin.data(), fin_ms.data(), *out, active);
  const auto t_run3 = std::chrono::steady_clock::now();
  long long chains = 0, wait = 0, pack = 0, launch = 0, unpack = 0;
  for (int l = 0; l < pl->L; ++l) {
    const PlanLane& ln = pl->lane[l];
    chains += ln.chains; wait += ln.wait_us; pack += ln.pack_us; launch += ln.launch_us; unpack += ln.unpack_us;
  }
  if (out->stats) { out->stats[5] = chains; out->stats[6] = wait; out->stats[7] = pl->L; }
  if (pl->trace)
    fprintf(stderr, "bp_plan host phases (%d lanes): pack %lld us, launch %lld us, wait %lld us, unpack %lld us over %lld rounds\n",
            pl->L, pack, launch, wait, unpack, chains);
  if (pl->trace)
    fprintf(stderr, "bp_plan host phases: load %.1f ms, gather %.1f ms, resume %.1f ms, store %.1f ms, run total %.1f ms\n",
            std::chrono::duration<double, std::milli>(t_run1 - t_run0).count(), st.gather_ms, st.resume_ms,
            std::chrono::duration<double, std::milli>(t_run3 - t_run2).count(),
            std::chrono::duration<double, std::milli>(t_run3 - t_run0).count());
  return 0;
}

extern "C" {

int bp_plan_run(bp_plan* pl, const bp_plan_in* in, bp_plan_out* out, void* stream) {
  return plan_run(pl, in, nullptr, out, stream);
}

int bp_plan_run_active(bp_plan* pl, const bp_plan_in* in, const int* active_host, bp_plan_out* out, void* stream) {
  return plan_run(pl, in, active_host, out, stream);
}

int bp_plan_destroy(bp_plan* pl) {
  if (!pl) return 0;
  pl->release();
  delete pl;
  return 0;
}

}  // extern "C"
