// engine.cu -- libgrove_place.so: host side of the placement engine and the C ABI of
// include/grove_place.h.  Everything that computes a placement runs in the kernels of kernels.cuh;
// the host sorts the topology once per label change, validates and uploads tables, and drives the
// relaxation rounds (relax.cuh).  There is no CPU fallback: without a CUDA device the engine cannot be created.
#include <omp.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdio>
#include <array>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <utility>
#include <new>
#include <numeric>
#include <string>
#include <vector>

#include "kernels.cuh"

using namespace grove;

namespace {

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
  ~DevBuf() { release(); }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  // grows geometrically: a pending set that creeps up tick after tick (churn) must not pay a cudaFree + cudaMalloc
  // of every table per cycle; falls back to the exact size when the padded one does not fit
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    const size_t want = std::max<size_t>(std::max<size_t>(n, (64u << 10) / sizeof(T)), cap + cap / 2);
    release();
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), want * sizeof(T));
    if (e == cudaSuccess) { cap = want; return e; }
    (void)cudaGetLastError();
    e = cudaMalloc(reinterpret_cast<void**>(&p), std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) cap = std::max<size_t>(n, 1); else p = nullptr;
    return e;
  }
};

template <typename T>
struct PinBuf {
  T* p = nullptr;
  size_t cap = 0;
  ~PinBuf() { if (p) cudaFreeHost(p); }
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    // pinned allocations cost milliseconds: start at 256 KB and double, so a growing pending set re-allocates rarely
    const size_t want = std::max<size_t>(std::max<size_t>(n, (256u << 10) / sizeof(T)), cap * 2);
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMallocHost(reinterpret_cast<void**>(&p), want * sizeof(T));
    if (e == cudaSuccess) cap = want; else p = nullptr;
    return e;
  }
};

// Size of the engine's host thread team (table validation, signature interning, staging copies).  One size for every
// parallel region: libgomp re-creates its team whenever the size changes.  Not taken from OMP_NUM_THREADS: launchers
// such as torchrun export OMP_NUM_THREADS=1 for every rank, which would serialise the per-cycle host work; the knob is
// GROVE_HOST_THREADS (default 8), capped by the processors this process may run on.
int host_threads() {
  static const int t = [] {
    int want = 8;
    if (const char* v = std::getenv("GROVE_HOST_THREADS")) want = std::atoi(v);
    return std::max(1, std::min(want, omp_get_num_procs()));
  }();
  return t;
}

// a host table the engine owns, in pinned memory: the caller's array is copied in once (by a few threads when it is
// large) and the upload from it is a plain asynchronous DMA
template <typename T>
struct PinVec {
  PinBuf<T> b;
  size_t n = 0;
  T& operator[](size_t i) { return b.p[i]; }
  const T& operator[](size_t i) const { return b.p[i]; }
  T* data() { return b.p; }
  cudaError_t assign(const T* src, size_t cnt) {
    cudaError_t e = b.ensure(cnt);
    if (e != cudaSuccess) return e;
    n = cnt;
    const size_t bytes = cnt * sizeof(T);
    // one team size for every parallel region of the engine: libgomp re-creates its thread team whenever the size changes
    const int T_ = bytes >= (256u << 10) ? host_threads() : 1;
#pragma omp parallel for num_threads(T_) schedule(static)
    for (int t = 0; t < T_; ++t) {
      const size_t a = bytes * t / T_, z = bytes * (t + 1) / T_;
      std::memcpy(reinterpret_cast<char*>(b.p) + a, reinterpret_cast<const char*>(src) + a, z - a);
    }
    return cudaSuccess;
  }
};

uint32_t fmix32(uint32_t x) {
  x = x * 0x9E3779B1u + 0x7F4A7C15u;
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}

}  // namespace

struct grove_engine {
  grove_config_t cfg{};
  std::string err;
  cudaStream_t stream = nullptr;
  cudaStream_t stream_score = nullptr;  // K2 runs beside the relaxation (they only share the fit data)
  cudaEvent_t ev_fit = nullptr, ev_score = nullptr, ev_s0 = nullptr, ev_s1 = nullptr;
  cudaEvent_t ev_nodes_up = nullptr, ev_tables_up = nullptr;  // the last upload out of the pinned node staging buffer / gang tables
  cudaEvent_t ev[10]{};

  // ---- topology (static until labels change) ----
  uint32_t N = 0, Npad = 0, L = 0, words = 0;
  std::vector<uint32_t> raw_dom;      // caller order, N * MAX_LEVELS: cache key
  std::vector<uint32_t> perm, inv;    // sorted <-> caller
  std::vector<uint32_t> tdom;         // sorted order, N * MAX_LEVELS tree-ified ids
  std::vector<uint8_t> vdepth;
  std::vector<uint32_t> dom_lo[GROVE_MAX_LEVELS], dom_hi[GROVE_MAX_LEVELS];
  uint32_t n_dom[GROVE_MAX_LEVELS]{}, unit[GROVE_MAX_LEVELS]{};
  DevBuf<grove_node_t> d_nodes_in;    // caller order, as loaded
  DevBuf<uint4> d_nres, d_ndom;
  DevBuf<uint32_t> d_perm, d_inv;
  DevBuf<uint8_t> d_vdepth;
  DevBuf<uint32_t> d_dom_lo[GROVE_MAX_LEVELS], d_dom_hi[GROVE_MAX_LEVELS], d_next_dom[GROVE_MAX_LEVELS];
  bool nodes_loaded = false;

  // ---- gang tables ----
  uint32_t G = 0, Q = 0, S = 0, P = 0;
  PinVec<grove_gang_t> gangs;
  PinVec<grove_clique_t> cliques;
  PinVec<grove_scope_t> scopes;
  PinBuf<uint8_t> h_state0;        // initial gang states of a cycle
  PinBuf<GangInfo> ginfo_pin;      // derived tables are built straight into pinned memory: their upload is a plain DMA
  PinBuf<CliqueInfo> cinfo_pin;
  PinBuf<uint32_t> by_rank_pin;
  PinBuf<uint32_t> shape_rep_pin;
  GangInfo* ginfo = nullptr;
  CliqueInfo* cinfo = nullptr;
  std::vector<uint4> sigs;
  uint32_t n_sigs = 0;
  bool gangs_loaded = false, ginfo_dirty = true;
  DevBuf<grove_gang_t> d_gangs;
  DevBuf<grove_clique_t> d_cliques;
  DevBuf<grove_scope_t> d_scopes;
  DevBuf<GangInfo> d_ginfo;
  DevBuf<CliqueInfo> d_cinfo;
  DevBuf<uint4> d_sigs;
  DevBuf<uint32_t> d_by_rank;
  std::vector<uint32_t> shape_rep;     // one representative gang per distinct gang shape
  uint32_t n_shapes = 0, pl_words = 0, pl_off[GROVE_MAX_LEVELS]{};
  bool shape_tables = false;
  DevBuf<uint32_t> d_shape_rep, d_shape_bits;

  // ---- relaxation state (relax.cuh) ----
  DevBuf<uint32_t> d_ctl, d_chg_round, d_eval_list, d_ent_node, d_cur_info, d_cur_glo, d_extent, d_sc_lo;
  DevBuf<uint32_t> d_nxt_node, d_nxt_info, d_nxt_glo, d_nxt_extent, d_nxt_sc_lo;
  DevBuf<uint32_t> d_rem_round, d_last_eval, d_fail_upto, d_nlive, d_ovf_head, d_ovf_next, d_add_stamp, d_rem_stamp, d_F, d_capsum, d_capmax, d_fin, d_totals;
  DevBuf<uint16_t> d_ent_meta, d_cur_n, d_nxt_meta, d_nxt_n;
  DevBuf<uint8_t> d_last_att, d_state, d_tstate, d_dirty, d_sc_lvl, d_nxt_tstate, d_nxt_sc_lvl, d_cap8, d_T;
  DevBuf<uint4> d_claims, d_ovf_claim;
  DevBuf<int4> d_ctot;
  DevBuf<uint32_t> d_cmaxr;
  DevBuf<grove_gang_status_t> d_status;
  DevBuf<grove_scope_status_t> d_scope_status;
  DevBuf<grove_placement_t> d_out;
  bool any_preferred = false;  // some gang / scope / clique carries a Preferred level
  uint32_t max_gang_pods = 0;
  uint32_t n_sm = 148;
  uint32_t cap_off[GROVE_MAX_LEVELS]{}, cap_stride = 0;
  bool dbg_on = false;
  DevBuf<uint32_t> d_dbg;
  uint32_t tune_window = 0;        // gangs beyond the settled prefix that relax concurrently (0: all)
  uint32_t tune_entry = 1024;      // gangs that may join the window per round (0: no limit)
  uint32_t tune_refresh = 1536;    // rebuild the capacity tables once the settled prefix has advanced this many gangs
  uint32_t tune_warp_ctas = 4;     // CTAs per SM of the warp-per-gang bookkeeping kernels (apply / detect / settle)
  uint32_t tune_batch = 3;         // rounds enqueued between two looks at the control words (GROVE_TUNE_AHEAD=0 / GROVE_DEBUG_ADMIT)
  uint32_t tune_ahead = 3;         // rounds kept in the queue while the host follows the relaxation through host-mapped progress words
  uint32_t tune_eval_ctas = 0;     // light k_eval warps per SM (0: 16)
  uint32_t tune_heavy_att = 4;     // a gang whose last evaluation made this many attempts is heavy: kW warps next time
  uint32_t tune_max_att = 3;       // a light (one-warp) evaluation gives up after this many attempts and comes back heavy
  uint32_t tune_heavy_ctas = 2;    // heavy-form CTAs per SM
  bool tune_overlap = true;        // K2 on a second stream beside the relaxation (GROVE_TUNE_OVERLAP=0 serialises them, e.g. to time K2 alone)
  bool tune_score = false;         // K2 score matrix: false = materialised on request (grove_build_score_matrix / the row getters),
                                   // true = every cycle, on the second stream beside the relaxation
  bool score_valid = false;        // d_T holds the matrix of the last cycle's start snapshot
  DevBuf<uint32_t> d_F0;           // K1 output over the cycle-start snapshot (the engine's own F follows the committed state)
  PinBuf<uint32_t> h_upd_idx;
  PinBuf<grove_node_t> h_upd_recs;
  cudaEvent_t ev_upd = nullptr;
  DevBuf<uint32_t> d_upd_idx;
  DevBuf<grove_node_t> d_upd_recs;
  DevBuf<grove_node_t> d_nodes_out;  // grove_get_nodes scratch
  PinBuf<uint32_t> h_ctl;
  uint32_t* h_live = nullptr;      // host-mapped words the last CTA of k_detect writes every round (round, front, done, refresh, ...):
  uint32_t* d_live = nullptr;      // the host follows the relaxation by reading memory, without a blocking call (grove_run_cycle)
  PinBuf<grove_gang_status_t> h_status;
  PinBuf<grove_scope_status_t> h_scope_status;
  PinBuf<grove_placement_t> h_out;
  PinBuf<grove_node_t> h_stage_nodes;
  uint32_t n_out = 0;
  bool have_results = false, have_scopes = false;
  grove_cycle_stats_t last{};

  bool in_cycle = false;
  uint64_t launches = 0;
  std::vector<grove_victim_t> victims;   // of the last grove_run_cycle_preempt
  // node-range shard of this handle (cfg.rank of cfg.world; the whole table when world <= 1): sorted node indices, cut at
  // top-level domain boundaries
  uint32_t shard_lo = 0, shard_hi = 0;
  bool score_pass_valid = false;   // the capacity tables + T describe the loaded snapshot (grove_run_score_pass)
  uint32_t t_c0 = 0, t_cpr = 0;    // ... and T holds the 16-node chunks [t_c0, t_c0 + t_cpr) of every row
  DevBuf<uint32_t> d_sig_sum;
};


#define CU_TRY(e, expr)                                                                       \
  do {                                                                                        \
    cudaError_t _c = (expr);                                                                  \
    if (_c != cudaSuccess) {                                                                  \
      (e)->err = std::string(#expr) + ": " + cudaGetErrorString(_c);                          \
      return _c == cudaErrorMemoryAllocation ? GROVE_ERR_OOM : GROVE_ERR_CUDA;                \
    }                                                                                         \
  } while (0)

static int32_t fail(grove_engine* e, int32_t code, const char* msg) { e->err = msg; return code; }

// Launch with programmatic stream serialization: the kernel's CTAs may become resident while the kernel before it on the
// stream is still running.  The kernel must call pdl_begin() (common.cuh) before it touches global memory.
template <typename... P, typename... A>
static cudaError_t launch_pdl(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, A&&... args) {
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...);
}

// ---------------------------------------------------------------------------------------------
// topology: sort by label path, tree-ify ids, domain ranges.  Host side; runs only when labels change.
// Restates what the reference hands a scheduler as the ordered level list
// (operator/internal/scheduler/kai/topology.go:103-135) plus the per-node label values.
// ---------------------------------------------------------------------------------------------
static int32_t build_topology(grove_engine* e, const grove_node_t* nodes, uint32_t n) {
  const uint32_t L = e->L;
  e->N = n;
  e->Npad = (n + 1023u) & ~1023u;
  e->words = e->Npad / 32;
  e->raw_dom.resize(size_t(n) * GROVE_MAX_LEVELS);
  for (uint32_t i = 0; i < n; ++i) std::memcpy(&e->raw_dom[size_t(i) * GROVE_MAX_LEVELS], nodes[i].dom, sizeof(uint32_t) * GROVE_MAX_LEVELS);
  e->perm.resize(n); e->inv.resize(n);
  std::iota(e->perm.begin(), e->perm.end(), 0u);
  const uint32_t* rd = e->raw_dom.data();
  std::sort(e->perm.begin(), e->perm.end(), [rd, L](uint32_t a, uint32_t b) {
    const uint32_t* x = rd + size_t(a) * GROVE_MAX_LEVELS; const uint32_t* y = rd + size_t(b) * GROVE_MAX_LEVELS;
    for (uint32_t l = 0; l < L; ++l) if (x[l] != y[l]) return x[l] < y[l];
    return a < b;
  });
  for (uint32_t i = 0; i < n; ++i) e->inv[e->perm[i]] = i;
  e->tdom.assign(size_t(e->Npad) * GROVE_MAX_LEVELS, GROVE_DOM_ABSENT);
  e->vdepth.assign(e->Npad, 0);
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) { e->dom_lo[l].clear(); e->dom_hi[l].clear(); e->n_dom[l] = 0; e->unit[l] = 0; }
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t* cur = rd + size_t(e->perm[i]) * GROVE_MAX_LEVELS;
    const uint32_t* prv = i ? rd + size_t(e->perm[i - 1]) * GROVE_MAX_LEVELS : nullptr;
    bool same_path = prv != nullptr;  // do cur and prv agree (and exist) on every level above l?
    uint32_t depth = 0;
    for (uint32_t l = 0; l < L; ++l) {
      if (cur[l] == GROVE_DOM_ABSENT) break;  // deeper labels are ignored once one is missing
      bool same = same_path && e->vdepth[i - 1] > l && prv[l] == cur[l];
      if (same) {
        uint32_t id = e->tdom[size_t(i - 1) * GROVE_MAX_LEVELS + l];
        e->tdom[size_t(i) * GROVE_MAX_LEVELS + l] = id;
        e->dom_hi[l][id] = i + 1;
      } else {
        e->tdom[size_t(i) * GROVE_MAX_LEVELS + l] = uint32_t(e->dom_lo[l].size());
        e->dom_lo[l].push_back(i); e->dom_hi[l].push_back(i + 1);
      }
      same_path = same;
      depth = l + 1;
    }
    e->vdepth[i] = uint8_t(depth);
  }
  for (uint32_t l = 0; l < L; ++l) {
    e->n_dom[l] = uint32_t(e->dom_lo[l].size());
    bool u = e->n_dom[l] > 0;
    for (uint32_t d = 0; d < e->n_dom[l] && u; ++d) u = (e->dom_hi[l][d] - e->dom_lo[l][d]) == 1;
    e->unit[l] = u ? 1u : 0u;
  }
  e->cap_stride = 0;
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) {
    e->cap_off[l] = e->cap_stride;
    if (l < L && !e->unit[l]) e->cap_stride += e->n_dom[l];
  }
  // upload static tables
  CU_TRY(e, e->d_perm.ensure(n)); CU_TRY(e, e->d_inv.ensure(n));
  CU_TRY(e, e->d_ndom.ensure(e->Npad)); CU_TRY(e, e->d_nres.ensure(e->Npad)); CU_TRY(e, e->d_vdepth.ensure(e->Npad));
  CU_TRY(e, cudaMemcpyAsync(e->d_perm.p, e->perm.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, e->stream));
  CU_TRY(e, cudaMemcpyAsync(e->d_inv.p, e->inv.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, e->stream));
  CU_TRY(e, cudaMemcpyAsync(e->d_ndom.p, e->tdom.data(), sizeof(uint4) * e->Npad, cudaMemcpyHostToDevice, e->stream));
  CU_TRY(e, cudaMemcpyAsync(e->d_vdepth.p, e->vdepth.data(), e->Npad, cudaMemcpyHostToDevice, e->stream));
  std::vector<uint32_t> nxt(size_t(n) + 1);
  for (uint32_t l = 0; l < L; ++l) {
    const uint32_t nd = e->n_dom[l];
    CU_TRY(e, e->d_dom_lo[l].ensure(nd)); CU_TRY(e, e->d_dom_hi[l].ensure(nd)); CU_TRY(e, e->d_next_dom[l].ensure(size_t(n) + 1));
    if (nd) {
      CU_TRY(e, cudaMemcpyAsync(e->d_dom_lo[l].p, e->dom_lo[l].data(), sizeof(uint32_t) * nd, cudaMemcpyHostToDevice, e->stream));
      CU_TRY(e, cudaMemcpyAsync(e->d_dom_hi[l].p, e->dom_hi[l].data(), sizeof(uint32_t) * nd, cudaMemcpyHostToDevice, e->stream));
    }
    uint32_t d = 0;
    for (uint32_t i = 0; i <= n; ++i) {  // first domain whose lo >= i
      while (d < nd && e->dom_lo[l][d] < i) ++d;
      nxt[i] = d;
    }
    CU_TRY(e, cudaMemcpyAsync(e->d_next_dom[l].p, nxt.data(), sizeof(uint32_t) * (size_t(n) + 1), cudaMemcpyHostToDevice, e->stream));
    CU_TRY(e, cudaStreamSynchronize(e->stream));  // nxt is reused
  }
  e->ginfo_dirty = true;
  // this handle's node-range shard: the top-level domains dealt out in order, as evenly as their sizes allow; nodes that lack
  // the top-level label (sorted last) go to the last rank
  {
    const uint32_t W = std::max<uint32_t>(e->cfg.world, 1u), R = e->cfg.world > 1 ? e->cfg.rank : 0u;
    auto cut = [&](uint32_t r) -> uint32_t {   // first node of rank r's shard
      if (r == 0) return 0u;
      if (r >= W) return n;
      const uint64_t target = uint64_t(n) * r / W;
      for (uint32_t d = 0; d < e->n_dom[0]; ++d) if (e->dom_lo[0][d] >= target) return e->dom_lo[0][d];
      return n;
    };
    e->shard_lo = cut(R); e->shard_hi = cut(R + 1);
  }
  return GROVE_OK;
}

static Topo make_topo(grove_engine* e) {
  Topo t{};
  t.nres = e->d_nres.p; t.ndom = e->d_ndom.p;
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) {
    t.dom_lo[l] = e->d_dom_lo[l].p; t.dom_hi[l] = e->d_dom_hi[l].p; t.next_dom[l] = e->d_next_dom[l].p;
    t.n_dom[l] = e->n_dom[l]; t.unit[l] = e->unit[l];
  }
  t.n = e->N; t.npad = e->Npad; t.L = e->L; t.words = e->words;
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) t.cap_off[l] = e->cap_off[l];
  t.cap_stride = e->cap_stride;
  return t;
}


static Tables make_tables(grove_engine* e) {
  Tables t{};
  t.gangs = e->d_gangs.p; t.cliques = e->d_cliques.p; t.scopes = e->d_scopes.p;
  t.ginfo = e->d_ginfo.p; t.cinfo = e->d_cinfo.p; t.sigs = e->d_sigs.p; t.by_rank = e->d_by_rank.p;
  t.G = e->G; t.Q = e->Q; t.S = e->n_sigs; t.NS = e->S;
  return t;
}

static Relax make_relax(grove_engine* e) {
  Relax r{};
  r.ctl = e->d_ctl.p; r.state = e->d_state.p; r.tstate = e->d_tstate.p; r.dirty = e->d_dirty.p; r.chg_round = e->d_chg_round.p;
  r.eval_list = e->d_eval_list.p; r.last_att = e->d_last_att.p;
  r.ent_node = e->d_ent_node.p; r.ent_meta = e->d_ent_meta.p; r.cur_n = e->d_cur_n.p; r.cur_info = e->d_cur_info.p; r.cur_glo = e->d_cur_glo.p;
  r.extent = e->d_extent.p; r.sc_lvl = e->d_sc_lvl.p; r.sc_lo = e->d_sc_lo.p;
  r.nxt_node = e->d_nxt_node.p; r.nxt_meta = e->d_nxt_meta.p; r.nxt_n = e->d_nxt_n.p; r.nxt_tstate = e->d_nxt_tstate.p;
  r.nxt_info = e->d_nxt_info.p; r.nxt_glo = e->d_nxt_glo.p; r.nxt_extent = e->d_nxt_extent.p; r.nxt_sc_lvl = e->d_nxt_sc_lvl.p; r.nxt_sc_lo = e->d_nxt_sc_lo.p;
  r.claims = e->d_claims.p; r.nlive = e->d_nlive.p; r.ovf_head = e->d_ovf_head.p; r.ovf_next = e->d_ovf_next.p; r.ovf_claim = e->d_ovf_claim.p;
  r.ovf_cap = uint32_t(std::min<size_t>(e->d_ovf_claim.cap, 0xFFFFFFF0u));
  r.ctot = e->d_ctot.p; r.cmaxr = e->d_cmaxr.p;
  r.add_stamp = e->d_add_stamp.p; r.rem_stamp = e->d_rem_stamp.p; r.rem_round = e->d_rem_round.p; r.last_eval = e->d_last_eval.p; r.fail_upto = e->d_fail_upto.p;
  r.F = e->d_F.p; r.cap8 = e->d_cap8.p; r.capsum = e->d_capsum.p; r.capmax = e->d_capmax.p; r.T = e->d_T.p;
  r.shape_bits = e->shape_tables ? e->d_shape_bits.p : nullptr; r.pl_words = e->pl_words;
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) r.pl_off[l] = e->pl_off[l];
  r.P = e->P; r.window = e->tune_window ? e->tune_window : (e->G ? e->G : 1u); r.entry = e->tune_entry ? e->tune_entry : r.window; r.heavy_att = e->tune_heavy_att;
  r.dbg = e->dbg_on ? e->d_dbg.p : nullptr;
  r.live = e->d_live;
  return r;
}

// ---------------------------------------------------------------------------------------------
extern "C" {

uint32_t grove_abi_version(void) { return GROVE_ABI_VERSION; }

const char* grove_last_error(grove_engine_t* e) { return e ? e->err.c_str() : "null engine"; }

int32_t grove_engine_create(const grove_config_t* cfg, grove_engine_t** out) {
  if (!cfg || !out) return GROVE_ERR_INVALID_ARG;
  *out = nullptr;
  if (cfg->abi_version != GROVE_ABI_VERSION) return GROVE_ERR_INVALID_ARG;
  if (cfg->n_levels < 1 || cfg->n_levels > GROVE_MAX_LEVELS) return GROVE_ERR_INVALID_ARG;
  if (cfg->world > 1 && cfg->rank >= cfg->world) return GROVE_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return GROVE_ERR_NO_DEVICE;  // no CPU fallback
  if (cfg->device < 0 || cfg->device >= ndev) return GROVE_ERR_NO_DEVICE;
  if (cudaSetDevice(cfg->device) != cudaSuccess) return GROVE_ERR_NO_DEVICE;
  grove_engine* e = new (std::nothrow) grove_engine();
  if (!e) return GROVE_ERR_OOM;
  e->cfg = *cfg; e->L = cfg->n_levels;
  { int sm = 0; if (cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, cfg->device) == cudaSuccess && sm > 0) e->n_sm = uint32_t(sm); }
  e->tune_window = cfg->window;
  if (const char* v = std::getenv("GROVE_TUNE_WINDOW")) if (!cfg->window) e->tune_window = uint32_t(std::max(0, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_ENTRY")) e->tune_entry = uint32_t(std::max(0, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_REFRESH")) e->tune_refresh = uint32_t(std::max(1, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_EVAL_CTAS")) e->tune_eval_ctas = uint32_t(std::max(1, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_WARP_CTAS")) e->tune_warp_ctas = uint32_t(std::max(1, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_BATCH")) e->tune_batch = uint32_t(std::max(1, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_AHEAD")) e->tune_ahead = uint32_t(std::max(0, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_HEAVY_ATT")) e->tune_heavy_att = uint32_t(std::max(1, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_MAX_ATT")) e->tune_max_att = uint32_t(std::max(0, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_HEAVY_CTAS")) e->tune_heavy_ctas = uint32_t(std::max(1, std::atoi(v)));
  if (const char* v = std::getenv("GROVE_TUNE_OVERLAP")) e->tune_overlap = std::atoi(v) != 0;
  if (const char* v = std::getenv("GROVE_TUNE_SCORE")) e->tune_score = std::atoi(v) != 0;
  if (std::getenv("GROVE_DEBUG_ADMIT")) e->dbg_on = true;
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);  // the latency-bound relaxation gets the SMs first
  if (cudaStreamCreateWithPriority(&e->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) { delete e; return GROVE_ERR_CUDA; }
  if (cudaStreamCreateWithPriority(&e->stream_score, cudaStreamNonBlocking, prio_lo) != cudaSuccess) { delete e; return GROVE_ERR_CUDA; }
  if (cudaFuncSetAttribute(k_eval<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kEvalSmem)) != cudaSuccess ||
      cudaFuncSetAttribute(k_eval<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kEvalSmem)) != cudaSuccess) { delete e; return GROVE_ERR_CUDA; }
  if (cudaEventCreateWithFlags(&e->ev_fit, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&e->ev_score, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_nodes_up, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&e->ev_tables_up, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_upd, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&e->ev_s0) != cudaSuccess || cudaEventCreate(&e->ev_s1) != cudaSuccess) { delete e; return GROVE_ERR_CUDA; }
  for (auto& ev : e->ev) if (cudaEventCreate(&ev) != cudaSuccess) { delete e; return GROVE_ERR_CUDA; }
  if (e->h_ctl.ensure(kCtlWords) != cudaSuccess) { delete e; return GROVE_ERR_OOM; }
  if (cudaHostAlloc(reinterpret_cast<void**>(&e->h_live), sizeof(uint32_t) * kLiveWords, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(reinterpret_cast<void**>(&e->d_live), e->h_live, 0) != cudaSuccess) { (void)cudaGetLastError(); e->h_live = nullptr; e->d_live = nullptr; }
  *out = e;
  return GROVE_OK;
}

void grove_engine_destroy(grove_engine_t* e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  cudaStreamSynchronize(e->stream);
  cudaStreamSynchronize(e->stream_score);
  for (auto& ev : e->ev) if (ev) cudaEventDestroy(ev);
  if (e->ev_s0) cudaEventDestroy(e->ev_s0);
  if (e->ev_s1) cudaEventDestroy(e->ev_s1);
  if (e->ev_fit) cudaEventDestroy(e->ev_fit);
  if (e->ev_nodes_up) cudaEventDestroy(e->ev_nodes_up);
  if (e->ev_tables_up) cudaEventDestroy(e->ev_tables_up);
  if (e->ev_upd) cudaEventDestroy(e->ev_upd);
  if (e->ev_score) cudaEventDestroy(e->ev_score);
  if (e->h_live) cudaFreeHost(e->h_live);
  if (e->stream_score) cudaStreamDestroy(e->stream_score);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}


static int32_t load_nodes_common(grove_engine* e, const grove_node_t* host_nodes, const void* dev_nodes, uint32_t n) {
  if (n == 0 || n > GROVE_MAX_NODES) return fail(e, GROVE_ERR_INVALID_ARG, "node count out of range");
  if (e->in_cycle) return fail(e, GROVE_ERR_STATE, "cycle in flight");
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  if (host_nodes) {
    CU_TRY(e, cudaEventSynchronize(e->ev_nodes_up));  // an earlier upload may still be reading the staging buffer
    CU_TRY(e, e->d_nodes_in.ensure(n));
    CU_TRY(e, e->h_stage_nodes.ensure(n));
    // one pass over the caller's snapshot by a few threads: copy to the pinned staging buffer (the caller's array is
    // not retained) and compare the labels with the cached topology's
    const bool cached = e->nodes_loaded && n == e->N;
    const int T = n >= 8192 ? host_threads() : 1;
    int differs = 0;
#pragma omp parallel for num_threads(T) schedule(static) reduction(| : differs)
    for (int t = 0; t < T; ++t) {
      const uint32_t a = uint32_t(uint64_t(n) * t / T), z = uint32_t(uint64_t(n) * (t + 1) / T);
      std::memcpy(e->h_stage_nodes.p + a, host_nodes + a, sizeof(grove_node_t) * (z - a));
      if (cached) {
        const uint32_t* rd = e->raw_dom.data();
        int d = 0;
        for (uint32_t i = a; i < z; ++i)
          d |= std::memcmp(rd + size_t(i) * GROVE_MAX_LEVELS, host_nodes[i].dom, sizeof(uint32_t) * GROVE_MAX_LEVELS) != 0;
        differs |= d;
      }
    }
    if (!cached || differs) { int32_t rc = build_topology(e, host_nodes, n); if (rc) return rc; }
    CU_TRY(e, cudaMemcpyAsync(e->d_nodes_in.p, e->h_stage_nodes.p, sizeof(grove_node_t) * n, cudaMemcpyHostToDevice, e->stream));
    CU_TRY(e, cudaEventRecord(e->ev_nodes_up, e->stream));
  } else {
    if (!e->nodes_loaded || n != e->N) return fail(e, GROVE_ERR_STATE, "device load needs a prior host load with the same labels");
    CU_TRY(e, cudaMemcpyAsync(e->d_nodes_in.p, dev_nodes, sizeof(grove_node_t) * n, cudaMemcpyDeviceToDevice, e->stream));
  }
  k_gather<<<(e->Npad + 255) / 256, 256, 0, e->stream>>>(e->d_nodes_in.p, e->d_perm.p, e->d_vdepth.p, e->d_nres.p, e->N, e->Npad);
  CU_TRY(e, cudaGetLastError());
  // (device source: read asynchronously on the engine's stream -- the header asks the caller to leave it alone until the next
  // blocking call on the handle returns; a synchronize here would cost every device-resident cycle a host round trip)
  e->nodes_loaded = true; e->score_pass_valid = false;
  return GROVE_OK;
}

int32_t grove_load_nodes(grove_engine_t* e, const grove_node_t* nodes, uint32_t n) {
  if (!e || !nodes) return GROVE_ERR_INVALID_ARG;
  return load_nodes_common(e, nodes, nullptr, n);
}

int32_t grove_load_nodes_device(grove_engine_t* e, const void* d_nodes, uint32_t n) {
  if (!e || !d_nodes) return GROVE_ERR_INVALID_ARG;
  return load_nodes_common(e, nullptr, d_nodes, n);
}

int32_t grove_update_nodes(grove_engine_t* e, const uint32_t* idx, const grove_node_t* recs, uint32_t n) {
  if (!e || (n && (!idx || !recs))) return GROVE_ERR_INVALID_ARG;
  if (!e->nodes_loaded) return fail(e, GROVE_ERR_STATE, "no node snapshot loaded");
  if (e->in_cycle) return fail(e, GROVE_ERR_STATE, "cycle in flight");
  if (n == 0) return GROVE_OK;
  e->score_pass_valid = false;
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  CU_TRY(e, cudaEventSynchronize(e->ev_upd));  // an earlier update may still be reading the pinned staging buffers
  CU_TRY(e, e->h_upd_idx.ensure(n)); CU_TRY(e, e->h_upd_recs.ensure(n));
  for (uint32_t i = 0; i < n; ++i) {
    if (idx[i] >= e->N) return fail(e, GROVE_ERR_INVALID_ARG, "node index out of range");
    if (std::memcmp(&e->raw_dom[size_t(idx[i]) * GROVE_MAX_LEVELS], recs[i].dom, sizeof(uint32_t) * GROVE_MAX_LEVELS) != 0)
      return fail(e, GROVE_ERR_INVALID_ARG, "grove_update_nodes cannot change labels; reload the snapshot");
    e->h_upd_idx.p[i] = e->inv[idx[i]];
  }
  std::memcpy(e->h_upd_recs.p, recs, sizeof(grove_node_t) * n);   // nothing of the caller's is referenced after return
  CU_TRY(e, e->d_upd_idx.ensure(n)); CU_TRY(e, e->d_upd_recs.ensure(n));
  CU_TRY(e, cudaMemcpyAsync(e->d_upd_idx.p, e->h_upd_idx.p, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, e->stream));
  CU_TRY(e, cudaMemcpyAsync(e->d_upd_recs.p, e->h_upd_recs.p, sizeof(grove_node_t) * n, cudaMemcpyHostToDevice, e->stream));
  CU_TRY(e, cudaEventRecord(e->ev_upd, e->stream));
  k_update<<<(n + 255) / 256, 256, 0, e->stream>>>(e->d_upd_idx.p, e->d_upd_recs.p, e->d_vdepth.p, e->d_perm.p, e->d_nres.p, e->d_nodes_in.p, n);
  CU_TRY(e, cudaGetLastError());
  return GROVE_OK;   // stream-ordered: the next call on this handle sees the update
}


int32_t grove_get_nodes(grove_engine_t* e, grove_node_t* out, uint32_t cap) {
  if (!e || !out) return GROVE_ERR_INVALID_ARG;
  if (!e->nodes_loaded) return fail(e, GROVE_ERR_STATE, "no node snapshot loaded");
  if (cap < e->N) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  CU_TRY(e, e->d_nodes_out.ensure(e->N));
  k_scatter<<<(e->N + 255) / 256, 256, 0, e->stream>>>(e->d_nodes_out.p, e->d_nodes_in.p, e->d_perm.p, e->d_nres.p, e->N);
  CU_TRY(e, cudaGetLastError());
  CU_TRY(e, cudaMemcpyAsync(out, e->d_nodes_out.p, sizeof(grove_node_t) * e->N, cudaMemcpyDeviceToHost, e->stream));
  CU_TRY(e, cudaStreamSynchronize(e->stream));
  return GROVE_OK;
}

// one gang; returns nullptr when it is well formed, else the reason (code through *code)
static const char* validate_gang(const grove_engine* e, const grove_gang_t* gangs, uint32_t G, const grove_clique_t* cliques, uint32_t Q,
                                 const grove_scope_t* scopes, uint32_t S, uint32_t gi, int32_t* code) {
  const uint32_t L = e->L;
  const grove_gang_t& g = gangs[gi];
  *code = GROVE_ERR_LIMIT;
  if (g.n_cliques == 0 || g.n_cliques > GROVE_MAX_GANG_CLIQUES) return "gang clique count out of range";
  if (g.n_scopes == 0 || g.n_scopes > GROVE_MAX_GANG_SCOPES) return "gang scope count out of range";
  *code = GROVE_ERR_INVALID_ARG;
  if (uint64_t(g.clique_off) + g.n_cliques > Q || uint64_t(g.scope_off) + g.n_scopes > S) return "gang table offsets out of range";
  if (g.level != GROVE_LEVEL_NONE && g.level >= L) return "gang level out of range";
  if (g.preferred != GROVE_LEVEL_NONE && (g.preferred >= L || (g.level != GROVE_LEVEL_NONE && g.preferred <= g.level)))
    return "gang preferred level must be a level deeper than the required one";
  if (g.anchor_node != GROVE_NONE_U32 && e->nodes_loaded && g.anchor_node >= e->N) return "anchor node out of range";
  if (g.base_gang != GROVE_NONE_U32 && (g.base_gang >= G || g.base_gang == gi)) return "base gang out of range";
  uint32_t pods = 0, next = 0;
  for (uint32_t si = 0; si < g.n_scopes; ++si) {
    const grove_scope_t& s = scopes[g.scope_off + si];
    if (s.first_clique != next || s.n_cliques == 0) return "scopes must tile the gang's cliques in order";
    if (s.level != GROVE_LEVEL_NONE && s.level >= L) return "scope level out of range";
    if (s.preferred1 && (s.preferred1 > L || (s.level != GROVE_LEVEL_NONE && uint32_t(s.preferred1) - 1u <= s.level)))
      return "scope preferred level must be a level deeper than the required one";
    if (next + s.n_cliques > g.n_cliques) return "scope exceeds gang";
    for (uint32_t i = 0; i < s.n_cliques; ++i) {
      const grove_clique_t& q = cliques[g.clique_off + next + i];
      if (GROVE_CLIQUE_SCOPE(q.scope) != si) return "clique.scope does not match its scope";
      if (q.level != GROVE_LEVEL_NONE && q.level >= L) return "clique level out of range";
      const uint32_t qp = GROVE_CLIQUE_PREFERRED(q.scope);
      if (qp != GROVE_LEVEL_NONE && (qp >= L || (q.level != GROVE_LEVEL_NONE && qp <= q.level)))
        return "clique preferred level must be a level deeper than the required one";
      if (q.replicas < q.min_replicas) return "replicas < min_replicas";
      pods += q.replicas;
    }
    next += s.n_cliques;
  }
  if (next != g.n_cliques) return "scopes do not cover the gang";
  if (pods > GROVE_MAX_GANG_PODS) { *code = GROVE_ERR_LIMIT; return "gang exceeds GROVE_MAX_GANG_PODS"; }
  return nullptr;
}

// same structural rules as the PodGang admission webhook guarantees
// (operator/internal/webhook/admission/pcs/validation/topologyconstraints.go:195-280); the first offending gang
// (lowest index) is reported whatever the thread count
static int32_t validate(grove_engine* e, const grove_gang_t* gangs, uint32_t G, const grove_clique_t* cliques, uint32_t Q,
                        const grove_scope_t* scopes, uint32_t S) {
  uint32_t first_bad = GROVE_NONE_U32;
  const int T = G >= 2048 ? host_threads() : 1;
#pragma omp parallel for num_threads(T) schedule(static) reduction(min : first_bad)
  for (uint32_t gi = 0; gi < G; ++gi) {
    int32_t code;
    if (gi < first_bad && validate_gang(e, gangs, G, cliques, Q, scopes, S, gi, &code)) first_bad = gi;
  }
  if (first_bad == GROVE_NONE_U32) return GROVE_OK;
  int32_t code = GROVE_ERR_INVALID_ARG;
  const char* why = validate_gang(e, gangs, G, cliques, Q, scopes, S, first_bad, &code);
  return fail(e, code, why ? why : "malformed gang tables");
}

int32_t grove_submit_gangs(grove_engine_t* e, const grove_gang_t* gangs, uint32_t n_gangs, const grove_clique_t* cliques,
                           uint32_t n_cliques, const grove_scope_t* scopes, uint32_t n_scopes) {
  if (!e || (n_gangs && (!gangs || !cliques || !scopes))) return GROVE_ERR_INVALID_ARG;
  if (e->in_cycle) return fail(e, GROVE_ERR_STATE, "cycle in flight");
  if (n_gangs >= (1u << 24)) return fail(e, GROVE_ERR_LIMIT, "too many gangs");  // order rank + round tag share a stamp word
  int32_t rc = validate(e, gangs, n_gangs, cliques, n_cliques, scopes, n_scopes);
  if (rc) return rc;
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  CU_TRY(e, cudaEventSynchronize(e->ev_tables_up));  // an earlier upload may still be reading the pinned tables
  e->G = n_gangs; e->Q = n_cliques; e->S = n_scopes;
  CU_TRY(e, e->gangs.assign(gangs, n_gangs));
  CU_TRY(e, e->cliques.assign(cliques, n_cliques));
  CU_TRY(e, e->scopes.assign(scopes, n_scopes));
  e->gangs_loaded = true; e->ginfo_dirty = true; e->have_results = false; e->score_pass_valid = false;
  bool pref = false;
  for (uint32_t g = 0; g < n_gangs && !pref; ++g) pref |= gangs[g].preferred != GROVE_LEVEL_NONE;
  for (uint32_t i = 0; i < n_scopes && !pref; ++i) pref |= scopes[i].preferred1 != 0;
  for (uint32_t i = 0; i < n_cliques && !pref; ++i) pref |= (cliques[i].scope >> 5) != 0;
  e->any_preferred = pref;
  CU_TRY(e, e->d_gangs.ensure(n_gangs)); CU_TRY(e, e->d_cliques.ensure(n_cliques)); CU_TRY(e, e->d_scopes.ensure(n_scopes));
  if (n_gangs) CU_TRY(e, cudaMemcpyAsync(e->d_gangs.p, e->gangs.data(), sizeof(grove_gang_t) * n_gangs, cudaMemcpyHostToDevice, e->stream));
  if (n_cliques) CU_TRY(e, cudaMemcpyAsync(e->d_cliques.p, e->cliques.data(), sizeof(grove_clique_t) * n_cliques, cudaMemcpyHostToDevice, e->stream));
  if (n_scopes) CU_TRY(e, cudaMemcpyAsync(e->d_scopes.p, e->scopes.data(), sizeof(grove_scope_t) * n_scopes, cudaMemcpyHostToDevice, e->stream));
  CU_TRY(e, cudaEventRecord(e->ev_tables_up, e->stream));
  return GROVE_OK;  // the uploads read engine-owned pinned memory: nothing of the caller's is referenced any more
}


// derived per-gang / per-clique tables: order rank, anchor (sorted index + ancestor ranges), entry slots
static int32_t build_ginfo(grove_engine* e) {
  const uint32_t G = e->G, Q = e->Q;
  const auto t_b0 = std::chrono::steady_clock::now();
  CU_TRY(e, e->ginfo_pin.ensure(G)); CU_TRY(e, e->cinfo_pin.ensure(Q)); CU_TRY(e, e->by_rank_pin.ensure(std::max<uint32_t>(G, 1)));
  e->ginfo = e->ginfo_pin.p; e->cinfo = e->cinfo_pin.p;
  {  // ginfo zeroed, cinfo all-ones (gang == NONE marks a row no gang owns yet), by the engine's thread team
    const int T0 = G >= 2048 ? host_threads() : 1;
#pragma omp parallel for num_threads(T0) schedule(static)
    for (int t = 0; t < T0; ++t) {
      const size_t g0 = size_t(G) * t / T0, g1 = size_t(G) * (t + 1) / T0, q0 = size_t(Q) * t / T0, q1 = size_t(Q) * (t + 1) / T0;
      std::memset(e->ginfo + g0, 0, sizeof(GangInfo) * (g1 - g0));
      std::memset(e->cinfo + q0, 0xFF, sizeof(CliqueInfo) * (q1 - q0));
    }
  }
  e->sigs.clear();
  const auto t_m0 = std::chrono::steady_clock::now();
  // order rank = position by (priority desc, index asc), and the anchors.  PriorityClasses are few: every thread counts
  // the distinct priorities of its gang range, one thread turns the counts into start offsets per (priority, thread),
  // and every thread numbers its own range -- a stable counting sort without the sorted array.
  bool bad_anchor = false;
  {
    constexpr size_t kMaxPrio = 64;
    const int T1 = G >= 2048 ? host_threads() : 1;
    std::vector<std::vector<std::pair<int32_t, uint32_t>>> seen(T1);   // per thread: (priority, count) in first-seen order
    std::vector<int32_t> prios;                                         // distinct, descending
    std::vector<uint32_t> start;                                        // [thread][priority index] first rank
    bool many = false;
#pragma omp parallel num_threads(T1)
    {
      const int t = omp_get_thread_num();
      const uint32_t g0 = uint32_t(uint64_t(G) * t / T1), g1 = uint32_t(uint64_t(G) * (t + 1) / T1);
      auto& mine = seen[t];
      bool over = false;
      for (uint32_t g = g0; g < g1 && !over; ++g) {
        const int32_t p = e->gangs[g].priority;
        size_t i = 0;
        while (i < mine.size() && mine[i].first != p) ++i;
        if (i == mine.size()) { if (mine.size() == kMaxPrio) { over = true; break; } mine.push_back({p, 0u}); }
        mine[i].second++;
      }
      if (over) {
#pragma omp atomic write
        many = true;
      }
#pragma omp barrier
#pragma omp single
      {
        for (const auto& v : seen) for (const auto& pc : v) prios.push_back(pc.first);
        std::sort(prios.begin(), prios.end(), std::greater<int32_t>());
        prios.erase(std::unique(prios.begin(), prios.end()), prios.end());
        if (prios.size() > kMaxPrio) many = true;
        if (!many) {
          start.assign(size_t(T1) * prios.size(), 0u);
          uint32_t run = 0;
          for (size_t k = 0; k < prios.size(); ++k)
            for (int tt = 0; tt < T1; ++tt) {
              start[size_t(tt) * prios.size() + k] = run;
              for (const auto& pc : seen[tt]) if (pc.first == prios[k]) run += pc.second;
            }
        }
      }  // implicit barrier
      bool bad = false;
      uint32_t next[kMaxPrio];
      if (!many) for (size_t k = 0; k < prios.size(); ++k) next[k] = start[size_t(t) * prios.size() + k];
      for (uint32_t gi = g0; gi < g1; ++gi) {
        const grove_gang_t& g = e->gangs[gi];
        if (!many) {
          size_t k = 0;
          while (prios[k] != g.priority) ++k;
          e->ginfo[gi].order = next[k]++;
        }
        if (g.anchor_node != GROVE_NONE_U32 && g.anchor_node >= e->N) { bad = true; continue; }
        e->ginfo[gi].anchor = g.anchor_node != GROVE_NONE_U32 ? e->inv[g.anchor_node] : fmix32(gi) % e->N;
      }
      if (bad) {
#pragma omp atomic write
        bad_anchor = true;
      }
    }
    if (many) {  // more distinct priorities than a scheduler has PriorityClasses: plain stable sort
      std::vector<uint32_t> ord(G);
      std::iota(ord.begin(), ord.end(), 0u);
      std::stable_sort(ord.begin(), ord.end(), [e](uint32_t a, uint32_t b) { return e->gangs[a].priority > e->gangs[b].priority; });
      for (uint32_t r = 0; r < G; ++r) e->ginfo[ord[r]].order = r;
    }
  }
  if (bad_anchor) return fail(e, GROVE_ERR_INVALID_ARG, "anchor node out of range");
  {  // the inverse: which gang has its turn at each rank
    const int T2 = G >= 2048 ? host_threads() : 1;
#pragma omp parallel for num_threads(T2) schedule(static)
    for (uint32_t gi = 0; gi < G; ++gi) e->by_rank_pin.p[e->ginfo[gi].order] = gi;
  }
  const auto t_m1 = std::chrono::steady_clock::now();
  // per-clique derived data + signature interning.  PodCliques stamped from one template (PCS / PCSG
  // replicas) share requests, selector class and binding depth: they share one fit-bitmap row.  Gang
  // ranges are processed by a few host threads with thread-local signature tables, merged afterwards.
  const auto t_m2 = std::chrono::steady_clock::now();
  struct SigTab {
    std::vector<std::array<uint32_t, 6>> tab = std::vector<std::array<uint32_t, 6>>(256, std::array<uint32_t, 6>{0, 0, 0, 0, 0, GROVE_NONE_U32});
    std::vector<std::array<uint32_t, 5>> keys;
    static uint32_t hash5(const std::array<uint32_t, 5>& k) { uint32_t h = k[0] * 0x9E3779B1u ^ k[1] * 0x85EBCA6Bu ^ (k[2] << 20) ^ (k[3] << 4) ^ k[4]; return h ^ (h >> 15); }
    uint32_t intern(const std::array<uint32_t, 5>& key) {
      if (keys.size() * 2 >= tab.size()) {
        std::vector<std::array<uint32_t, 6>> nt(tab.size() * 4, std::array<uint32_t, 6>{0, 0, 0, 0, 0, GROVE_NONE_U32});
        for (const auto& r : tab) if (r[5] != GROVE_NONE_U32) {
          size_t h = hash5({r[0], r[1], r[2], r[3], r[4]}) & (nt.size() - 1);
          while (nt[h][5] != GROVE_NONE_U32) h = (h + 1) & (nt.size() - 1);
          nt[h] = r;
        }
        tab.swap(nt);
      }
      size_t h = hash5(key) & (tab.size() - 1);
      while (tab[h][5] != GROVE_NONE_U32 && !(tab[h][0] == key[0] && tab[h][1] == key[1] && tab[h][2] == key[2] && tab[h][3] == key[3] && tab[h][4] == key[4]))
        h = (h + 1) & (tab.size() - 1);
      if (tab[h][5] == GROVE_NONE_U32) { tab[h] = {key[0], key[1], key[2], key[3], key[4], uint32_t(keys.size())}; keys.push_back(key); }
      return tab[h][5];
    }
  };
  const int T = G >= 2048 ? host_threads() : 1;
  std::vector<SigTab> local(T);
  std::vector<uint32_t> gang_pods(G, 0);
  int shared_rows = 0;
#pragma omp parallel num_threads(T) reduction(+ : shared_rows)
  {
    const int t = omp_get_thread_num();
    const uint32_t g0 = uint32_t(uint64_t(G) * t / T), g1 = uint32_t(uint64_t(G) * (t + 1) / T);
    SigTab& st = local[t];
    for (uint32_t gi = g0; gi < g1; ++gi) {
      const grove_gang_t& g = e->gangs[gi];
      uint32_t pods = 0;
      for (uint32_t si = 0; si < g.n_scopes; ++si) {
        const grove_scope_t& s = e->scopes[g.scope_off + si];
        for (uint32_t i = 0; i < s.n_cliques; ++i) {
          const uint32_t qi = g.clique_off + s.first_clique + i;
          const grove_clique_t& q = e->cliques[qi];
          uint32_t nd = 0;
          if (g.level != GROVE_LEVEL_NONE) nd = std::max(nd, uint32_t(g.level) + 1);
          if (s.level != GROVE_LEVEL_NONE) nd = std::max(nd, uint32_t(s.level) + 1);
          if (q.level != GROVE_LEVEL_NONE) nd = std::max(nd, uint32_t(q.level) + 1);
          if (e->cinfo[qi].gang != GROVE_NONE_U32) shared_rows++;  // rows of different threads never overlap unless the tables are malformed
          e->cinfo[qi] = CliqueInfo{gi, nd, st.intern({q.req_cpu_milli, q.req_mem_mib, q.req_gpu, q.class_mask, nd}), uint32_t(t)};
          pods += q.replicas;
        }
      }
      gang_pods[gi] = pods;
    }
  }
  const auto t_m3 = std::chrono::steady_clock::now();
  if (shared_rows) return fail(e, GROVE_ERR_INVALID_ARG, "clique rows shared between gangs");
  SigTab global;
  std::vector<std::vector<uint32_t>> remap(T);
  for (int t = 0; t < T; ++t) { remap[t].resize(local[t].keys.size()); for (size_t k = 0; k < local[t].keys.size(); ++k) remap[t][k] = global.intern(local[t].keys[k]); }
  e->sigs.resize(global.keys.size());
  for (size_t k = 0; k < global.keys.size(); ++k) { const auto& key = global.keys[k]; e->sigs[k] = make_uint4(key[0], key[1], key[2], key[3] | (key[4] << 16)); }
  // thread-local signature ids -> global ids (pad carried the id of the thread that interned the row)
#pragma omp parallel for num_threads(T) schedule(static)
  for (uint32_t qi = 0; qi < Q; ++qi)
    if (e->cinfo[qi].gang != GROVE_NONE_U32) { e->cinfo[qi].sig = remap[e->cinfo[qi].pad][e->cinfo[qi].sig]; e->cinfo[qi].pad = 0; }
  // Gang SHAPES: what the candidate pre-filter of a gang depends on is its structure (levels, scopes, per-clique
  // signature / MinReplicas / level), not its anchor or rank.  PodGangs stamped from one template share a shape, so the
  // pre-filter is evaluated once per (shape, candidate domain) per capacity-table build (k_shape_plaus) instead of once
  // per (gang evaluation, candidate).  Interned like the signatures: thread-local tables over gang ranges, merged.
  {
    auto shape_hash = [e](uint32_t gi) {
      const grove_gang_t& g = e->gangs[gi];
      uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t(g.n_cliques) << 32 | uint64_t(g.n_scopes) << 16 | uint64_t(g.level) << 8 | g.preferred);
      auto mix = [&h](uint64_t v) { h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2); };
      for (uint32_t si = 0; si < g.n_scopes; ++si) { const grove_scope_t& s = e->scopes[g.scope_off + si]; mix(uint64_t(s.first_clique) | uint64_t(s.n_cliques) << 16 | uint64_t(s.level) << 32 | uint64_t(s.preferred1) << 40); }
      for (uint32_t c = 0; c < g.n_cliques; ++c) { const grove_clique_t& q = e->cliques[g.clique_off + c]; mix(uint64_t(e->cinfo[g.clique_off + c].sig) | uint64_t(q.min_replicas) << 32 | uint64_t(q.level) << 40 | uint64_t(q.scope) << 48); }
      return h;
    };
    auto shape_equal = [e](uint32_t a, uint32_t b) {
      const grove_gang_t& x = e->gangs[a]; const grove_gang_t& y = e->gangs[b];
      if (x.n_cliques != y.n_cliques || x.n_scopes != y.n_scopes || x.level != y.level || x.preferred != y.preferred) return false;
      for (uint32_t si = 0; si < x.n_scopes; ++si) {
        const grove_scope_t& s = e->scopes[x.scope_off + si]; const grove_scope_t& t = e->scopes[y.scope_off + si];
        if (s.first_clique != t.first_clique || s.n_cliques != t.n_cliques || s.level != t.level || s.preferred1 != t.preferred1) return false;
      }
      for (uint32_t c = 0; c < x.n_cliques; ++c) {
        const grove_clique_t& q = e->cliques[x.clique_off + c]; const grove_clique_t& r = e->cliques[y.clique_off + c];
        if (e->cinfo[x.clique_off + c].sig != e->cinfo[y.clique_off + c].sig || q.min_replicas != r.min_replicas || q.level != r.level || q.scope != r.scope) return false;
      }
      return true;
    };
    struct ShapeTab {   // open addressing on the hash; value = representative gang
      std::vector<std::pair<uint64_t, uint32_t>> tab = std::vector<std::pair<uint64_t, uint32_t>>(256, {0, GROVE_NONE_U32});
      std::vector<uint32_t> reps;
      size_t used = 0;
    };
    auto intern = [&](ShapeTab& st, uint32_t gi, uint64_t h) -> uint32_t {   // -> index into st.reps
      if (st.used * 2 >= st.tab.size()) {
        std::vector<std::pair<uint64_t, uint32_t>> nt(st.tab.size() * 4, {0, GROVE_NONE_U32});
        for (const auto& r : st.tab) if (r.second != GROVE_NONE_U32) { size_t k = r.first & (nt.size() - 1); while (nt[k].second != GROVE_NONE_U32) k = (k + 1) & (nt.size() - 1); nt[k] = r; }
        st.tab.swap(nt);
      }
      size_t k = h & (st.tab.size() - 1);
      while (st.tab[k].second != GROVE_NONE_U32 && !(st.tab[k].first == h && shape_equal(st.reps[st.tab[k].second], gi))) k = (k + 1) & (st.tab.size() - 1);
      if (st.tab[k].second == GROVE_NONE_U32) { st.tab[k] = {h, uint32_t(st.reps.size())}; st.reps.push_back(gi); st.used++; }
      return st.tab[k].second;
    };
    std::vector<ShapeTab> lsh(T);
    std::vector<uint32_t> lid(G);
#pragma omp parallel num_threads(T)
    {
      const int t = omp_get_thread_num();
      const uint32_t g0 = uint32_t(uint64_t(G) * t / T), g1 = uint32_t(uint64_t(G) * (t + 1) / T);
      for (uint32_t gi = g0; gi < g1; ++gi) lid[gi] = intern(lsh[t], gi, shape_hash(gi));
    }
    ShapeTab gsh;
    std::vector<std::vector<uint32_t>> smap(T);
    for (int t = 0; t < T; ++t) { smap[t].resize(lsh[t].reps.size()); for (size_t k = 0; k < lsh[t].reps.size(); ++k) smap[t][k] = intern(gsh, lsh[t].reps[k], shape_hash(lsh[t].reps[k])); }
    e->shape_rep = gsh.reps;
    e->n_shapes = uint32_t(gsh.reps.size());
#pragma omp parallel num_threads(T)
    {
      const int t = omp_get_thread_num();
      const uint32_t g0 = uint32_t(uint64_t(G) * t / T), g1 = uint32_t(uint64_t(G) * (t + 1) / T);
      for (uint32_t gi = g0; gi < g1; ++gi) e->ginfo[gi].pad = smap[t][lid[gi]];
    }
    // bit layout of one shape's row: every level's domains, each level padded to a word
    uint32_t bits = 0;
    for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) { e->pl_off[l] = bits; if (l < e->L) bits += (e->n_dom[l] + 31u) & ~31u; }
    e->pl_words = bits / 32;
    // worth it while the rows stay small next to the work they save; otherwise every evaluation runs the pre-filter itself
    e->shape_tables = e->n_shapes && uint64_t(e->n_shapes) * e->pl_words * 4 <= (256ull << 20) && e->n_shapes <= G / 2 + 16;
  }
  uint32_t pod_off = 0;
  e->max_gang_pods = 0;
  for (uint32_t gi = 0; gi < G; ++gi) { e->ginfo[gi].pod_off = pod_off; pod_off += gang_pods[gi]; e->max_gang_pods = std::max(e->max_gang_pods, gang_pods[gi]); }
  e->P = pod_off;
  const auto t_b1 = std::chrono::steady_clock::now();
  for (uint32_t qi = 0; qi < Q; ++qi)
    if (e->cinfo[qi].gang == GROVE_NONE_U32) return fail(e, GROVE_ERR_INVALID_ARG, "clique row owned by no gang");
  e->n_sigs = uint32_t(e->sigs.size());
  CU_TRY(e, e->d_ginfo.ensure(G)); CU_TRY(e, e->d_cinfo.ensure(Q)); CU_TRY(e, e->d_sigs.ensure(e->n_sigs));
  CU_TRY(e, e->d_by_rank.ensure(std::max<uint32_t>(G, 1)));
  if (e->n_sigs) CU_TRY(e, cudaMemcpyAsync(e->d_sigs.p, e->sigs.data(), sizeof(uint4) * e->n_sigs, cudaMemcpyHostToDevice, e->stream));
  if (G) {
    CU_TRY(e, cudaMemcpyAsync(e->d_ginfo.p, e->ginfo, sizeof(GangInfo) * G, cudaMemcpyHostToDevice, e->stream));
    k_anchor<<<(G + 255) / 256, 256, 0, e->stream>>>(make_topo(e), e->d_ginfo.p, G);  // ancestor ranges from the device-resident tree
    CU_TRY(e, cudaGetLastError());
  }
  if (Q) CU_TRY(e, cudaMemcpyAsync(e->d_cinfo.p, e->cinfo, sizeof(CliqueInfo) * Q, cudaMemcpyHostToDevice, e->stream));
  if (G) CU_TRY(e, cudaMemcpyAsync(e->d_by_rank.p, e->by_rank_pin.p, sizeof(uint32_t) * G, cudaMemcpyHostToDevice, e->stream));
  if (e->shape_tables) {
    CU_TRY(e, e->d_shape_rep.ensure(e->n_shapes)); CU_TRY(e, e->d_shape_bits.ensure(size_t(e->n_shapes) * e->pl_words));
    CU_TRY(e, e->shape_rep_pin.ensure(e->n_shapes));   // (pinned: the upload is a plain DMA the host does not wait for; the buffer is
    std::memcpy(e->shape_rep_pin.p, e->shape_rep.data(), sizeof(uint32_t) * e->n_shapes);   //  rewritten only after the cycle that reads it)
    CU_TRY(e, cudaMemcpyAsync(e->d_shape_rep.p, e->shape_rep_pin.p, sizeof(uint32_t) * e->n_shapes, cudaMemcpyHostToDevice, e->stream));
  }
  e->ginfo_dirty = false;
  if (std::getenv("GROVE_DEBUG_HOST")) {
    const auto t_b2 = std::chrono::steady_clock::now();
    auto us = [](auto a, auto b) { return (long)std::chrono::duration_cast<std::chrono::microseconds>(b - a).count(); };
    std::fprintf(stderr, "build_ginfo: tables %ld us (init %ld, order %ld, anchors %ld, cliques %ld, merge %ld), upload %ld us\n", us(t_b0, t_b1), us(t_b0, t_m0), us(t_m0, t_m1), us(t_m1, t_m2), us(t_m2, t_m3), us(t_m3, t_b1), us(t_b1, t_b2));
  }
  return GROVE_OK;
}

// words of the per-domain capacity sum / max tables (each): k_fit accumulates into them with atomics, so the kernel before it
// (k_reset for the first build of a cycle, k_fold for the others) zeroes them
static uint32_t cap_words(const grove_engine* e) { return e->n_sigs * e->cap_stride; }

// capacity tables over the committed state: K1 fit bitmap for every signature, per-node capacities, per-domain sum / max
static int32_t build_cap_tables(grove_engine* e, const Topo& tp, const Tables& tb, const Relax& rx) {
  if (!e->n_sigs) return GROVE_OK;
  dim3 gfit(e->Npad / 1024, std::min<uint32_t>((e->n_sigs + kFitTile - 1) / kFitTile, 65535u));
  CU_TRY(e, launch_pdl(k_fit, gfit, 1024, 0, e->stream, tp, tb, e->d_F.p, e->d_cap8.p, e->cap_stride ? e->d_capsum.p : nullptr,
                       e->cap_stride ? e->d_capmax.p : nullptr));
  CU_TRY(e, launch_pdl(k_clear_stale, (e->Npad / 4 + 255) / 256, 256, 0, e->stream, rx, e->Npad / 4));
  if (e->shape_tables) {   // the candidate pre-filter of every gang shape over every domain of its candidate levels
    // only the levels some shape takes its candidates from (Preferred down to Required): a CTA that has nothing to do still
    // costs its launch, and the unit level alone would be tens of thousands of them
    uint32_t mx = 0;
    for (uint32_t i = 0; i < e->n_shapes; ++i) {
      const grove_gang_t& g = e->gangs[e->shape_rep[i]];
      const int base = g.level != GROVE_LEVEL_NONE ? int(g.level) : -1;
      const int first = g.preferred != GROVE_LEVEL_NONE && int(g.preferred) > base ? int(g.preferred) : base;
      for (int l = std::max(base, 0); l <= first && l < int(e->L); ++l) mx = std::max(mx, e->n_dom[l]);
    }
    if (mx) CU_TRY(e, launch_pdl(k_shape_plaus, dim3((mx + 31) / 32, e->n_shapes, e->L), 128, 0, e->stream, tp, tb, rx, e->d_shape_rep.p));
    e->launches += 1;
  }
  CU_TRY(e, cudaGetLastError());
  e->launches += 2;
  return GROVE_OK;
}

static int32_t cycle_begin(grove_engine* e) {
  if (!e->nodes_loaded) return fail(e, GROVE_ERR_STATE, "no node snapshot loaded");
  if (!e->gangs_loaded) return fail(e, GROVE_ERR_STATE, "no gangs submitted");
  if (e->in_cycle) return fail(e, GROVE_ERR_STATE, "cycle in flight");
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  if (e->ginfo_dirty) { int32_t rc = build_ginfo(e); if (rc) return rc; }
  const uint32_t G = e->G, Q = e->Q, S = e->S, P = e->P, N = e->Npad;
  const size_t g1 = std::max<uint32_t>(G, 1), p1 = std::max<uint32_t>(P, 1), s1 = std::max<uint32_t>(S, 1);
  CU_TRY(e, e->d_ctl.ensure(kCtlWords));
  CU_TRY(e, e->d_state.ensure(g1)); CU_TRY(e, e->d_tstate.ensure(g1)); CU_TRY(e, e->d_dirty.ensure(g1)); CU_TRY(e, e->d_chg_round.ensure(g1));
  CU_TRY(e, e->d_eval_list.ensure(g1)); CU_TRY(e, e->d_last_att.ensure(g1));
  CU_TRY(e, e->d_ent_node.ensure(p1)); CU_TRY(e, e->d_ent_meta.ensure(p1)); CU_TRY(e, e->d_cur_n.ensure(g1)); CU_TRY(e, e->d_cur_info.ensure(g1));
  CU_TRY(e, e->d_cur_glo.ensure(g1)); CU_TRY(e, e->d_extent.ensure(g1)); CU_TRY(e, e->d_sc_lvl.ensure(s1)); CU_TRY(e, e->d_sc_lo.ensure(s1));
  CU_TRY(e, e->d_nxt_node.ensure(p1)); CU_TRY(e, e->d_nxt_meta.ensure(p1)); CU_TRY(e, e->d_nxt_n.ensure(g1)); CU_TRY(e, e->d_nxt_tstate.ensure(g1));
  CU_TRY(e, e->d_nxt_info.ensure(g1)); CU_TRY(e, e->d_nxt_glo.ensure(g1)); CU_TRY(e, e->d_nxt_extent.ensure(g1));
  CU_TRY(e, e->d_nxt_sc_lvl.ensure(s1)); CU_TRY(e, e->d_nxt_sc_lo.ensure(s1));
  CU_TRY(e, e->d_claims.ensure(size_t(N) * kClaimSlots)); CU_TRY(e, e->d_nlive.ensure(N / 4)); CU_TRY(e, e->d_ovf_head.ensure(N));
  CU_TRY(e, e->d_ovf_next.ensure(4 * p1 + 1024)); CU_TRY(e, e->d_ovf_claim.ensure(4 * p1 + 1024));
  CU_TRY(e, e->d_ctot.ensure(N)); CU_TRY(e, e->d_cmaxr.ensure(N));
  CU_TRY(e, e->d_add_stamp.ensure(N)); CU_TRY(e, e->d_rem_stamp.ensure(e->words)); CU_TRY(e, e->d_rem_round.ensure(e->words));
  CU_TRY(e, e->d_last_eval.ensure(g1)); CU_TRY(e, e->d_fail_upto.ensure(g1));
  CU_TRY(e, e->d_status.ensure(g1)); CU_TRY(e, e->d_scope_status.ensure(s1)); CU_TRY(e, e->d_out.ensure(p1));
  CU_TRY(e, e->h_status.ensure(g1)); CU_TRY(e, e->h_scope_status.ensure(s1)); CU_TRY(e, e->h_out.ensure(p1));
  CU_TRY(e, e->d_fin.ensure((G + kFinThreads - 1) / kFinThreads + 4)); CU_TRY(e, e->d_totals.ensure(4));
  // the S x N tables and the Q x N score matrix
  {
    const size_t fw = size_t(e->n_sigs) * e->words, cb = size_t(e->n_sigs) * N, tw = size_t(e->n_sigs) * std::max<uint32_t>(e->cap_stride, 1);
    if (e->d_F.ensure(std::max<size_t>(fw, 1)) != cudaSuccess || e->d_cap8.ensure(std::max<size_t>(cb, 1)) != cudaSuccess ||
        e->d_capsum.ensure(tw) != cudaSuccess || e->d_capmax.ensure(tw) != cudaSuccess ||
        (e->tune_score && e->d_T.ensure(std::max<size_t>(size_t(Q) * N, 1)) != cudaSuccess)) {
      (void)cudaGetLastError();
      return fail(e, GROVE_ERR_OOM, "fit / capacity / score matrices do not fit in device memory");
    }
  }
  if (e->dbg_on) { CU_TRY(e, e->d_dbg.ensure(g1 * 8 + 8)); CU_TRY(e, cudaMemsetAsync(e->d_dbg.p, 0, g1 * 32 + 32, e->stream)); }
  {
    const uint32_t W = e->tune_window ? e->tune_window : std::max(G, 1u);
    const uint32_t E = e->tune_entry ? e->tune_entry : W;
    if (e->h_live) { std::memset(e->h_live, 0, sizeof(uint32_t) * kLiveWords); e->h_live[kLiveRound] = 1; }
    k_reset<<<e->n_sm * 4, 256, 0, e->stream>>>(make_relax(e), G, S, N, e->words, std::min(G, std::min(W, E)), cap_words(e));
    CU_TRY(e, cudaGetLastError());
  }
  e->launches = 0; e->in_cycle = true; e->have_results = false; e->have_scopes = false;
  e->victims.clear(); e->score_pass_valid = false;
  std::memset(&e->last, 0, sizeof(e->last));
  return GROVE_OK;
}

static int32_t finish_cycle(grove_engine* e) {
  const Topo tp = make_topo(e); const Tables tb = make_tables(e); const Relax rx = make_relax(e);
  const uint32_t G = e->G;
  e->n_out = 0;
  if (G) {
    const uint32_t ncta = (G + kFinThreads - 1) / kFinThreads;
    CU_TRY(e, cudaMemsetAsync(e->d_fin.p + ncta, 0, sizeof(uint32_t) * 4, e->stream));
    CU_TRY(e, launch_pdl(k_fin_count, ncta, kFinThreads, 0, e->stream, tb, rx, e->d_fin.p));
    CU_TRY(e, launch_pdl(k_fin_scan, 1, 1024, 0, e->stream, e->d_fin.p, ncta, e->d_totals.p));
    CU_TRY(e, launch_pdl(k_fin_status, ncta, kFinThreads, 0, e->stream, tb, rx, e->d_fin.p, e->d_perm.p, e->d_status.p));
    CU_TRY(e, launch_pdl(k_emit, (G * 32 + 255) / 256, 256, 0, e->stream, tb, rx, e->d_perm.p, e->d_status.p, e->d_out.p, e->d_scope_status.p));
    CU_TRY(e, cudaGetLastError());
    e->launches += 4;
    CU_TRY(e, cudaMemcpyAsync(e->h_ctl.p, e->d_totals.p, sizeof(uint32_t) * 4, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(e, cudaMemcpyAsync(e->h_status.p, e->d_status.p, sizeof(grove_gang_status_t) * G, cudaMemcpyDeviceToHost, e->stream));
    // the placement count is only known on the device: copy the upper bound's worth in the same breath when it is small,
    // else wait for the count
    const bool eager = size_t(e->P) * sizeof(grove_placement_t) <= (8u << 20);   // a few hundred KB at C4: cheaper than a second round trip
    if (eager && e->P) CU_TRY(e, cudaMemcpyAsync(e->h_out.p, e->d_out.p, sizeof(grove_placement_t) * e->P, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    e->n_out = e->h_ctl.p[0];
    if (!eager) {
      if (e->n_out) CU_TRY(e, cudaMemcpyAsync(e->h_out.p, e->d_out.p, sizeof(grove_placement_t) * e->n_out, cudaMemcpyDeviceToHost, e->stream));
      CU_TRY(e, cudaStreamSynchronize(e->stream));
    }
    e->last.gangs_admitted = e->h_ctl.p[1]; e->last.gangs_rejected = e->h_ctl.p[2];
  }
  (void)tp;
  e->last.pods_bound = e->n_out; e->last.kernel_launches = e->launches;
  e->have_results = true; e->in_cycle = false;
  return GROVE_OK;
}

struct CycleGuard {   // every error exit of a cycle leaves the handle usable (ADVICE round 1: in_cycle stayed set)
  grove_engine* e; bool armed = true;
  ~CycleGuard() { if (armed) { e->in_cycle = false; cudaStreamSynchronize(e->stream); cudaStreamSynchronize(e->stream_score); } }
};

int32_t grove_run_cycle(grove_engine_t* e, grove_cycle_stats_t* stats) {
  if (!e) return GROVE_ERR_INVALID_ARG;
  int32_t rc = cycle_begin(e);
  if (rc) return rc;
  CycleGuard guard{e};
  const Topo tp = make_topo(e); const Tables tb = make_tables(e); const Relax rx = make_relax(e);
  const uint32_t G = e->G;
  CU_TRY(e, cudaEventRecord(e->ev[8], e->stream));
  uint32_t rounds = 0;
  if (G) {
    // K1 + capacity tables over the cycle-start snapshot; K2 (score matrix) forks to the second stream
    CU_TRY(e, cudaEventRecord(e->ev[0], e->stream));
    rc = build_cap_tables(e, tp, tb, rx);
    if (rc) return rc;
    CU_TRY(e, cudaEventRecord(e->ev[1], e->stream));
    CU_TRY(e, e->d_F0.ensure(std::max<size_t>(size_t(e->n_sigs) * e->words, 1)));
    CU_TRY(e, cudaMemcpyAsync(e->d_F0.p, e->d_F.p, sizeof(uint32_t) * size_t(e->n_sigs) * e->words, cudaMemcpyDeviceToDevice, e->stream));
    e->score_valid = false;
    if (e->tune_score && e->Q) {
      cudaStream_t ss = e->tune_overlap ? e->stream_score : e->stream;
      if (e->tune_overlap) CU_TRY(e, cudaEventRecord(e->ev_fit, e->stream));
      if (e->tune_overlap) CU_TRY(e, cudaStreamWaitEvent(ss, e->ev_fit, 0));
      CU_TRY(e, cudaEventRecord(e->ev_s0, ss));
      k_score<<<dim3(1, std::min<uint32_t>(e->Q, 65535u)), 256, 0, ss>>>(tp, tb, e->d_F0.p, e->d_T.p, e->Q, 0u, e->Npad >> 4, size_t(e->Npad));  // one CTA per row
      e->score_valid = true;
      CU_TRY(e, cudaEventRecord(e->ev_s1, ss));
      if (e->tune_overlap) CU_TRY(e, cudaEventRecord(e->ev_score, e->stream_score));
      e->launches += 1;
    }
    CU_TRY(e, cudaEventRecord(e->ev[2], e->stream));
    const uint32_t W = rx.window;
    const uint32_t per_sm = e->tune_eval_ctas ? e->tune_eval_ctas : 16u;   // light warps
    const uint32_t light_ctas = (std::max(1u, std::min(W, e->n_sm * per_sm)) + kHeavyWarps - 1) / kHeavyWarps;
    const uint32_t heavy_ctas = std::max(1u, std::min(W, e->n_sm * e->tune_heavy_ctas));
    const uint32_t warp_ctas = std::max(1u, std::min((W * 32 + 255) / 256, e->n_sm * e->tune_warp_ctas));
    // Rounds are enqueued `batch` at a time without waiting: every kernel returns at once when the cycle is over, so the
    // host only looks at the control words between batches (to rebuild the capacity tables when the settled prefix has
    // moved on, and to know when to stop).  GROVE_DEBUG_ADMIT looks after every round.
    const uint32_t batch = e->dbg_on ? 1u : std::max(1u, e->tune_batch);
    uint32_t next_round = 1;   // number of the next round to be enqueued (rounds advance one by one until the cycle is over)
    auto enqueue_round = [&]() -> int32_t {
      if (next_round > 1 && next_round % kTagRounds == 0) {   // the stamp tags wrap: forget the stamps of the epoch that ends
        CU_TRY(e, cudaMemsetAsync(e->d_add_stamp.p, 0xFF, sizeof(uint32_t) * e->Npad, e->stream));
        CU_TRY(e, cudaMemsetAsync(e->d_rem_stamp.p, 0xFF, sizeof(uint32_t) * e->words, e->stream));
      }
      // heavy gangs (head of the list) kHeavyWarps warps each, light gangs (tail) a warp each: one launch, two roles
      CU_TRY(e, launch_pdl(e->any_preferred ? k_eval<true> : k_eval<false>, heavy_ctas + light_ctas, kEvalThreads, kEvalSmem, e->stream,
                           tp, tb, rx, heavy_ctas, e->tune_max_att));
      CU_TRY(e, launch_pdl(k_apply, warp_ctas, 256, 0, e->stream, tb, rx));
      CU_TRY(e, launch_pdl(k_detect, warp_ctas, 256, 0, e->stream, tp, tb, rx, e->tune_refresh));
      e->launches += 3;
      ++next_round;
      return GROVE_OK;
    };
    // the final gangs' claims -> committed state (relax.cuh k_fold); before a rebuild it also zeroes the capacity sums / maxima
    auto fold = [&](bool rebuild) -> int32_t {
      CU_TRY(e, launch_pdl(k_fold, warp_ctas, 256, 0, e->stream, tb, rx, e->d_nres.p, rebuild ? cap_words(e) : 0u));
      e->launches += 1;
      return GROVE_OK;
    };
    auto fold_and_rebuild = [&]() -> int32_t { int32_t r = fold(true); return r ? r : build_cap_tables(e, tp, tb, rx); };
    // Following the relaxation WITHOUT blocking calls: the last CTA of k_detect leaves (round, done, refresh, ...) in host-mapped
    // memory; the host keeps `ahead` rounds enqueued beyond the one that runs and adds one more each time it sees a round end
    // (or a table rebuild first, when the device asked for one).  The GPU never waits for the host; the only waste is the
    // <= ahead rounds in the queue when the cycle ends, which return at once.
    const bool polled = e->h_live && e->tune_ahead > 0 && !e->dbg_on;
    bool use_batch = !polled;   // the batch protocol below: also the way out should the progress words ever stop moving
    if (polled) {
      volatile uint32_t* lv = e->h_live;
      uint32_t enq = 0, rebuild_at = 0;   // rounds enqueued; the last rebuild enqueued runs before round rebuild_at + 1
      for (; enq < e->tune_ahead; ++enq) { rc = enqueue_round(); if (rc) return rc; }
      CU_TRY(e, cudaGetLastError());
      uint64_t spins = 0;
      for (;;) {
        const uint32_t completed = lv[kLiveRound] - 1u;
        if (lv[kLiveDone] && completed >= 1u) break;
        if (completed + e->tune_ahead > enq) {   // fewer than `ahead` rounds in flight: top the queue up
          if (lv[kLiveRefresh] && completed > rebuild_at) { rc = fold_and_rebuild(); if (rc) return rc; rebuild_at = enq; }   // (the flag is fresh again once round rebuild_at + 1 has ended)
          rc = enqueue_round(); if (rc) return rc;
          ++enq; spins = 0;
          continue;
        }
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();   // (a polite spin: the sibling hyper-thread may be another rank's)
#endif
        if ((++spins & 0xFFFFu) == 0) {   // a failed launch / a sticky error must not leave the host spinning
          const cudaError_t q = cudaStreamQuery(e->stream);
          if (q != cudaSuccess && q != cudaErrorNotReady) { e->err = std::string("relaxation: ") + cudaGetErrorString(q); return GROVE_ERR_CUDA; }
          // nothing left in flight on the engine's stream, yet the words say rounds are outstanding: do not trust them any
          // further -- the control words themselves are read from here on
          if (q == cudaSuccess && lv[kLiveRound] - 1u == completed && !lv[kLiveDone]) { use_batch = true; break; }
        }
      }
    }
    for (; use_batch;) {   // (the batch protocol: look at the control words between batches of rounds)
      for (uint32_t b = 0; b < batch; ++b) { rc = enqueue_round(); if (rc) return rc; }
      CU_TRY(e, cudaGetLastError());
      CU_TRY(e, cudaMemcpyAsync(e->h_ctl.p, e->d_ctl.p, sizeof(uint32_t) * kCtlWords, cudaMemcpyDeviceToHost, e->stream));
      CU_TRY(e, cudaStreamSynchronize(e->stream));
      const uint32_t* c = e->h_ctl.p;
      rounds = c[kRound] - 1;
      if (e->dbg_on) {
        std::fprintf(stderr, "round %u: front %u hi %u evals so far %u ovf %u\n", rounds, c[kFront], c[kHi], c[kEvals], c[kOvfCount]);
        std::vector<uint32_t> h(size_t(G) * 8); std::vector<uint8_t> ts(G);
        cudaMemcpy(h.data(), e->d_dbg.p, h.size() * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(ts.data(), e->d_tstate.p, G, cudaMemcpyDeviceToHost);
        std::vector<uint32_t> idx;
        for (uint32_t g = 0; g < G; ++g) if (h[size_t(g) * 8 + 7] == rounds) idx.push_back(g);
        std::sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) { return h[size_t(a) * 8 + 4] > h[size_t(b) * 8 + 4]; });
        uint64_t cyc = 0; for (uint32_t g : idx) cyc += h[size_t(g) * 8 + 4];
        std::fprintf(stderr, "  %zu packed evals, mean %.0f cyc, median %u; slowest:", idx.size(), idx.empty() ? 0.0 : double(cyc) / idx.size(), idx.empty() ? 0u : h[size_t(idx[idx.size() / 2]) * 8 + 4]);
        for (size_t i = 0; i < std::min<size_t>(idx.size(), 6); ++i) {
          const uint32_t g = idx[i]; const uint32_t* d = &h[size_t(g) * 8];
          std::fprintf(stderr, " [g%u rank%u st%u scopes%u: %u cyc, %u plaus, %u att]", g, e->ginfo[g].order, unsigned(ts[g]), unsigned(e->gangs[g].n_scopes), d[4], d[6], d[5]);
        }
        std::fprintf(stderr, "\n");
      }
      if (c[kOvfCount] > rx.ovf_cap) return fail(e, GROVE_ERR_LIMIT, "claim overflow pool exhausted");
      if (c[kDone]) break;
      if (c[kRefresh]) { rc = fold_and_rebuild(); if (rc) return rc; }
    }
    if (polled && !use_batch) {   // the cycle is over (the queue holds at most a few rounds that return at once): the final control words
      CU_TRY(e, cudaMemcpyAsync(e->h_ctl.p, e->d_ctl.p, sizeof(uint32_t) * kCtlWords, cudaMemcpyDeviceToHost, e->stream));
      CU_TRY(e, cudaStreamSynchronize(e->stream));
      if (e->h_ctl.p[kOvfCount] > rx.ovf_cap) return fail(e, GROVE_ERR_LIMIT, "claim overflow pool exhausted");
      rounds = e->h_ctl.p[kRound] - 1;
    }
    rc = fold(false); if (rc) return rc;   // everything is final now: the committed state and the final states of the outputs
    e->last.evaluations = e->h_ctl.p[kEvals];
  }
  CU_TRY(e, cudaEventRecord(e->ev[3], e->stream));
  if (e->tune_score && e->tune_overlap && G && e->Q) CU_TRY(e, cudaStreamWaitEvent(e->stream, e->ev_score, 0));  // the cycle ends when K2 has too
  rc = finish_cycle(e);
  if (rc) return rc;
  CU_TRY(e, cudaEventRecord(e->ev[9], e->stream));
  CU_TRY(e, cudaEventSynchronize(e->ev[9]));
  guard.armed = false;
  float t = 0;
  if (G) {
    cudaEventElapsedTime(&t, e->ev[0], e->ev[1]); e->last.ms_fit = t;
    if (e->tune_score && e->Q) { cudaEventElapsedTime(&t, e->ev_s0, e->ev_s1); e->last.ms_score = t; }
    cudaEventElapsedTime(&t, e->ev[2], e->ev[3]); e->last.ms_admit = t;
  }
  cudaEventElapsedTime(&t, e->ev[3], e->ev[9]); e->last.ms_commit = t;
  cudaEventElapsedTime(&t, e->ev[8], e->ev[9]); e->last.ms_total = t;
  e->last.rounds = rounds;
  e->last.pairs_evaluated = uint64_t(e->tune_score ? e->Q : e->n_sigs) * e->N;   // K1 works per signature, K2 per clique
  if (e->dbg_on && G) {
    std::vector<uint32_t> h(size_t(G) * 8 + 8);
    cudaMemcpy(h.data(), e->d_dbg.p, h.size() * 4, cudaMemcpyDeviceToHost);
    { const uint32_t* w = &h[size_t(G) * 8];
      std::fprintf(stderr, "warp 0 of every evaluation: %u evals, %.0f cyc each; %u staged attempts: staging %.0f cyc, sub-domain pre-filter %.0f, packing %.0f per attempt\n",
                   w[5], w[5] ? double(w[4]) / w[5] : 0.0, w[3], w[3] ? double(w[0]) / w[3] : 0.0, w[3] ? double(w[1]) / w[3] : 0.0, w[3] ? double(w[2]) / w[3] : 0.0);
      std::fprintf(stderr, "  of the staging: claim lines %.0f cyc, overflow chains %.0f per attempt\n", w[3] ? double(w[6]) / w[3] : 0.0, w[3] ? double(w[7]) / w[3] : 0.0); }
    uint64_t ev = 0, pl = 0, at = 0, mx = 0;
    for (uint32_t g = 0; g < G; ++g) { ev += h[g * 8]; pl += h[g * 8 + 1]; at += h[g * 8 + 2]; mx = std::max<uint64_t>(mx, h[g * 8]); }
    std::fprintf(stderr, "cycle: %u rounds, %llu evaluations (max %llu per gang), plausible/eval %.1f, attempts/eval %.2f\n", rounds,
                 (unsigned long long)ev, (unsigned long long)mx, ev ? double(pl) / ev : 0.0, ev ? double(at) / ev : 0.0);
  }
  if (stats) *stats = e->last;
  return GROVE_OK;
}

int32_t grove_get_placements(grove_engine_t* e, grove_placement_t* out, uint32_t cap, uint32_t* n_out) {
  if (!e || !n_out) return GROVE_ERR_INVALID_ARG;
  if (!e->have_results) return fail(e, GROVE_ERR_STATE, "no completed cycle");
  *n_out = e->n_out;
  if (!out) return GROVE_OK;
  if (cap < e->n_out) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  std::memcpy(out, e->h_out.p, sizeof(grove_placement_t) * e->n_out);
  return GROVE_OK;
}

int32_t grove_get_gang_status(grove_engine_t* e, grove_gang_status_t* out, uint32_t cap) {
  if (!e || !out) return GROVE_ERR_INVALID_ARG;
  if (!e->have_results) return fail(e, GROVE_ERR_STATE, "no completed cycle");
  if (cap < e->G) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  std::memcpy(out, e->h_status.p, sizeof(grove_gang_status_t) * e->G);
  return GROVE_OK;
}

int32_t grove_get_scope_domains(grove_engine_t* e, grove_scope_status_t* out, uint32_t cap) {
  if (!e || !out) return GROVE_ERR_INVALID_ARG;
  if (!e->have_results) return fail(e, GROVE_ERR_STATE, "no completed cycle");
  if (cap < e->S) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  if (!e->have_scopes && e->S) {   // fetched on demand: most callers only bind pods
    CU_TRY(e, cudaSetDevice(e->cfg.device));
    CU_TRY(e, cudaMemcpyAsync(e->h_scope_status.p, e->d_scope_status.p, sizeof(grove_scope_status_t) * e->S, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    e->have_scopes = true;
  }
  std::memcpy(out, e->h_scope_status.p, sizeof(grove_scope_status_t) * e->S);
  return GROVE_OK;
}

// K2 over the snapshot the last cycle started from: T[q][n] = fit ? 1 + closeness(n, anchor of q's gang) : 0.  The admission
// derives its visiting order from the anchor's ancestor ranges and never reads this matrix, so it is materialised on
// request (a scheduler that wants per-node scores -- the Score extension point -- asks for it); GROVE_TUNE_SCORE=1 builds
// it every cycle instead, on a second stream beside the relaxation.  *ms (nullable) = device time of the kernel.
int32_t grove_build_score_matrix(grove_engine_t* e, float* ms) {
  if (!e) return GROVE_ERR_INVALID_ARG;
  if (!e->have_results) return fail(e, GROVE_ERR_STATE, "no completed cycle");
  if (ms) *ms = 0.f;
  if (e->Q == 0) return GROVE_OK;
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  if (e->score_valid && !ms) return GROVE_OK;
  if (e->d_T.ensure(size_t(e->Q) * e->Npad) != cudaSuccess) { (void)cudaGetLastError(); return fail(e, GROVE_ERR_OOM, "score matrix does not fit in device memory"); }
  const Topo tp = make_topo(e); const Tables tb = make_tables(e);
  CU_TRY(e, cudaEventRecord(e->ev_s0, e->stream));
  k_score<<<dim3(1, std::min<uint32_t>(e->Q, 65535u)), 256, 0, e->stream>>>(tp, tb, e->d_F0.p, e->d_T.p, e->Q, 0u, e->Npad >> 4, size_t(e->Npad));  // one CTA per row
  CU_TRY(e, cudaGetLastError());
  CU_TRY(e, cudaEventRecord(e->ev_s1, e->stream));
  CU_TRY(e, cudaEventSynchronize(e->ev_s1));
  float t = 0; cudaEventElapsedTime(&t, e->ev_s0, e->ev_s1);
  e->last.ms_score = t; e->score_valid = true;
  if (ms) *ms = t;
  return GROVE_OK;
}

// ---------------------------------------------------------------------------------------------
// Reclaim pass (include/grove_place.h "preemption / reclaim"; DESIGN.md section 1).  Host orchestration around the same
// device path: the gangs the ordinary pass rejected are re-submitted priority class by priority class (descending) against
// the reclaim view of that class -- the evaluation of a gang does not depend on WHICH running gangs end up evicted, only on
// what is free plus what is evictable, so a whole class is one ordinary cycle on the augmented node table; the victims
// are then chosen gang by gang in order, exactly as the sequential statement says.
// ---------------------------------------------------------------------------------------------
namespace {
struct Res { int64_t cpu = 0, mem = 0, gpu = 0, pods = 0; };
inline bool covers(const grove_node_t& n, const Res& r) {
  return int64_t(n.free_cpu_milli) >= r.cpu && int64_t(n.free_mem_mib) >= r.mem && int64_t(n.free_gpu) >= r.gpu && int64_t(n.free_pods) >= r.pods;
}
inline void give(grove_node_t& n, const grove_holding_t& h) {
  n.free_cpu_milli += h.cpu_milli; n.free_mem_mib += h.mem_mib; n.free_gpu = uint16_t(n.free_gpu + h.gpu); n.free_pods = uint16_t(n.free_pods + h.pods);
}
}  // namespace

int32_t grove_run_cycle_preempt(grove_engine_t* e, const grove_running_gang_t* running, uint32_t n_running,
                                const grove_holding_t* holdings, uint32_t n_holdings, grove_cycle_stats_t* stats) {
  if (!e || (n_running && !running) || (n_holdings && !holdings)) return GROVE_ERR_INVALID_ARG;
  for (uint32_t r = 0; r < n_running; ++r)
    if (uint64_t(running[r].holding_off) + running[r].n_holdings > n_holdings) return fail(e, GROVE_ERR_INVALID_ARG, "running gang holdings out of range");
  if (e->nodes_loaded) for (uint32_t h = 0; h < n_holdings; ++h)
    if (holdings[h].node >= e->N) return fail(e, GROVE_ERR_INVALID_ARG, "holding on a node out of range");
  grove_cycle_stats_t st0{};
  int32_t rc = grove_run_cycle(e, &st0);
  if (rc) return rc;
  const uint32_t G = e->G, Q = e->Q, S = e->S, N = e->N;
  // the ordinary pass's outputs and the submission itself (the handle is re-used for the class cycles)
  std::vector<grove_gang_t> gangs(e->gangs.data(), e->gangs.data() + G);
  std::vector<grove_clique_t> cliques(e->cliques.data(), e->cliques.data() + Q);
  std::vector<grove_scope_t> scopes(e->scopes.data(), e->scopes.data() + S);
  std::vector<grove_gang_status_t> status(e->h_status.p, e->h_status.p + G);
  std::vector<grove_placement_t> place(e->h_out.p, e->h_out.p + e->n_out);
  std::vector<grove_scope_status_t> sstat(std::max<uint32_t>(S, 1));
  if (S) { rc = grove_get_scope_domains(e, sstat.data(), S); if (rc) return rc; }
  std::vector<int32_t> classes;
  for (uint32_t g = 0; g < G; ++g) if (status[g].state == GROVE_GANG_REJECTED) classes.push_back(gangs[g].priority);
  std::sort(classes.begin(), classes.end(), std::greater<int32_t>());
  classes.erase(std::unique(classes.begin(), classes.end()), classes.end());
  int32_t min_run = INT32_MAX;
  for (uint32_t r = 0; r < n_running; ++r) min_run = std::min(min_run, running[r].priority);
  std::vector<grove_victim_t> victims;
  std::vector<std::vector<grove_placement_t>> extra(G);   // placements of the preemptors, by gang
  if (!classes.empty() && n_running && classes.front() > min_run) {
    std::vector<grove_node_t> real(N), view(N);
    rc = grove_get_nodes(e, real.data(), N);
    if (rc) return rc;
    // whatever goes wrong from here on, the handle goes back to the caller's submission on the node table of the ordinary pass
    // (its class cycles re-use the handle); the error of the failing call is what the caller sees
    struct Restore {
      grove_engine* e; const std::vector<grove_node_t>* nodes; const std::vector<grove_gang_t>* g; const std::vector<grove_clique_t>* c; const std::vector<grove_scope_t>* s; bool armed = true;
      ~Restore() {
        if (!armed) return;
        const std::string keep = e->err;
        grove_load_nodes(e, nodes->data(), uint32_t(nodes->size()));
        grove_submit_gangs(e, g->data(), uint32_t(g->size()), c->data(), uint32_t(c->size()), s->data(), uint32_t(s->size()));
        e->err = keep;
      }
    };
    const std::vector<grove_node_t> real0 = real;
    Restore restore{e, &real0, &gangs, &cliques, &scopes};
    std::vector<uint8_t> evicted(n_running, 0);
    // running gangs by node (CSR), for the victim choice
    std::vector<uint32_t> at_off(size_t(N) + 1, 0), at_run(n_holdings);
    for (uint32_t r = 0; r < n_running; ++r) for (uint32_t h = 0; h < running[r].n_holdings; ++h) ++at_off[holdings[running[r].holding_off + h].node + 1];
    for (uint32_t n = 0; n < N; ++n) at_off[n + 1] += at_off[n];
    { std::vector<uint32_t> cur(at_off.begin(), at_off.end() - 1);
      for (uint32_t r = 0; r < n_running; ++r) for (uint32_t h = 0; h < running[r].n_holdings; ++h) at_run[cur[holdings[running[r].holding_off + h].node]++] = r; }
    for (int32_t p : classes) {
      bool any = false;
      view = real;
      for (uint32_t r = 0; r < n_running; ++r) {
        if (evicted[r] || running[r].priority >= p) continue;
        any = true;
        for (uint32_t h = 0; h < running[r].n_holdings; ++h) give(view[holdings[running[r].holding_off + h].node], holdings[running[r].holding_off + h]);
      }
      if (!any) continue;   // nothing to reclaim for this class (nor for the lower ones)
      // the class's rejected gangs as a submission of their own: anchors pinned to what the ordinary pass used, no gating
      // (a rejected gang's base gang, if any, was admitted before it)
      std::vector<uint32_t> ids;
      std::vector<grove_gang_t> sg; std::vector<grove_clique_t> sq; std::vector<grove_scope_t> ss;
      for (uint32_t g = 0; g < G; ++g) {
        if (status[g].state != GROVE_GANG_REJECTED || gangs[g].priority != p) continue;
        grove_gang_t x = gangs[g];
        if (x.anchor_node == GROVE_NONE_U32) x.anchor_node = e->perm[fmix32(g) % N];
        x.base_gang = GROVE_NONE_U32;
        x.clique_off = uint32_t(sq.size()); x.scope_off = uint32_t(ss.size());
        sq.insert(sq.end(), cliques.begin() + gangs[g].clique_off, cliques.begin() + gangs[g].clique_off + gangs[g].n_cliques);
        ss.insert(ss.end(), scopes.begin() + gangs[g].scope_off, scopes.begin() + gangs[g].scope_off + gangs[g].n_scopes);
        ids.push_back(g); sg.push_back(x);
      }
      if (ids.empty()) continue;
      rc = grove_load_nodes(e, view.data(), N); if (rc) return rc;
      rc = grove_submit_gangs(e, sg.data(), uint32_t(sg.size()), sq.data(), uint32_t(sq.size()), ss.data(), uint32_t(ss.size())); if (rc) return rc;
      grove_cycle_stats_t stp{};
      rc = grove_run_cycle(e, &stp); if (rc) return rc;
      st0.rounds += stp.rounds; st0.evaluations += stp.evaluations; st0.kernel_launches += stp.kernel_launches;
      st0.ms_fit += stp.ms_fit; st0.ms_admit += stp.ms_admit; st0.ms_commit += stp.ms_commit; st0.ms_total += stp.ms_total;
      std::vector<grove_scope_status_t> ssp(std::max<size_t>(ss.size(), 1));
      if (!ss.empty()) { rc = grove_get_scope_domains(e, ssp.data(), uint32_t(ss.size())); if (rc) return rc; }
      for (uint32_t k = 0; k < ids.size(); ++k) {   // sub-submission order == order rank (one priority)
        const grove_gang_status_t& sp = e->h_status.p[k];
        if (sp.state != GROVE_GANG_ADMITTED) continue;
        const uint32_t g = ids[k];
        // what the gang puts on each node, nodes in the order its placement first names them
        std::vector<uint32_t> order; std::vector<Res> use;
        for (uint32_t i = 0; i < sp.n_pods; ++i) {
          const grove_placement_t pl = e->h_out.p[sp.placement_off + i];
          const grove_clique_t& q = sq[pl.clique];
          size_t j = 0;
          for (; j < order.size(); ++j) if (order[j] == pl.node) break;
          if (j == order.size()) { order.push_back(pl.node); use.emplace_back(); }
          use[j].cpu += q.req_cpu_milli; use[j].mem += q.req_mem_mib; use[j].gpu += q.req_gpu; use[j].pods += 1;
          extra[g].push_back(grove_placement_t{gangs[g].clique_off + (pl.clique - sg[k].clique_off), pl.node});
        }
        for (size_t j = 0; j < order.size(); ++j) {
          const uint32_t n = order[j];
          while (!covers(real[n], use[j])) {
            uint32_t v = GROVE_NONE_U32;   // lowest priority first, then the highest running index
            for (uint32_t a = at_off[n]; a < at_off[n + 1]; ++a) {
              const uint32_t r = at_run[a];
              if (evicted[r] || running[r].priority >= p) continue;
              if (v == GROVE_NONE_U32 || running[r].priority < running[v].priority || (running[r].priority == running[v].priority && r > v)) v = r;
            }
            if (v == GROVE_NONE_U32) return fail(e, GROVE_ERR_STATE, "reclaim pass: a preemptor's node cannot be freed");
            evicted[v] = 1;
            for (uint32_t h = 0; h < running[v].n_holdings; ++h) give(real[holdings[running[v].holding_off + h].node], holdings[running[v].holding_off + h]);
            victims.push_back(grove_victim_t{v, g});
          }
          real[n].free_cpu_milli -= uint32_t(use[j].cpu); real[n].free_mem_mib -= uint32_t(use[j].mem);
          real[n].free_gpu = uint16_t(real[n].free_gpu - use[j].gpu); real[n].free_pods = uint16_t(real[n].free_pods - use[j].pods);
        }
        grove_gang_status_t o = sp;
        o.reserved0 = GROVE_STATUS_PREEMPTOR;
        status[g] = o;   // placement_off is assigned when the outputs are merged
        for (uint32_t si = 0; si < gangs[g].n_scopes; ++si) sstat[gangs[g].scope_off + si] = ssp[sg[k].scope_off + si];
        st0.gangs_admitted += 1; st0.gangs_rejected -= 1;
      }
    }
    // the handle goes back to the caller's submission, on the node table that is really free now
    restore.armed = false;
    rc = grove_load_nodes(e, real.data(), N); if (rc) return rc;
    rc = grove_submit_gangs(e, gangs.data(), G, cliques.data(), Q, scopes.data(), S); if (rc) return rc;
  }
  // merged outputs: placements grouped by gang in submission order
  CU_TRY(e, e->h_status.ensure(std::max<uint32_t>(G, 1))); CU_TRY(e, e->h_scope_status.ensure(std::max<uint32_t>(S, 1)));
  size_t total = 0;
  for (uint32_t g = 0; g < G; ++g) total += status[g].state == GROVE_GANG_ADMITTED ? status[g].n_pods : 0u;
  CU_TRY(e, e->h_out.ensure(std::max<size_t>(total, 1)));
  std::vector<grove_placement_t> merged; merged.reserve(total);
  for (uint32_t g = 0; g < G; ++g) {
    if (status[g].state != GROVE_GANG_ADMITTED) continue;
    const uint32_t off = uint32_t(merged.size());
    if (status[g].reserved0 & GROVE_STATUS_PREEMPTOR) merged.insert(merged.end(), extra[g].begin(), extra[g].end());
    else merged.insert(merged.end(), place.begin() + status[g].placement_off, place.begin() + status[g].placement_off + status[g].n_pods);
    status[g].placement_off = off;
  }
  std::memcpy(e->h_out.p, merged.data(), sizeof(grove_placement_t) * merged.size());
  std::memcpy(e->h_status.p, status.data(), sizeof(grove_gang_status_t) * G);
  if (S) std::memcpy(e->h_scope_status.p, sstat.data(), sizeof(grove_scope_status_t) * S);
  e->n_out = uint32_t(merged.size());
  st0.pods_bound = e->n_out;
  e->last = st0;
  e->victims = std::move(victims);
  e->have_results = true; e->have_scopes = true; e->score_valid = false;
  if (stats) *stats = st0;
  return GROVE_OK;
}

int32_t grove_get_victims(grove_engine_t* e, grove_victim_t* out, uint32_t cap, uint32_t* n_out) {
  if (!e || !n_out) return GROVE_ERR_INVALID_ARG;
  if (!e->have_results) return fail(e, GROVE_ERR_STATE, "no completed cycle");
  *n_out = uint32_t(e->victims.size());
  if (!out) return GROVE_OK;
  if (cap < e->victims.size()) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  std::memcpy(out, e->victims.data(), sizeof(grove_victim_t) * e->victims.size());
  return GROVE_OK;
}

// ---------------------------------------------------------------------------------------------
// Multi-GPU score pass (BASELINE.json north_star: "the node-state table shards across GPUs only when the synthetic cluster
// exceeds single-GPU capacity, with one NCCL all-reduce over NVLink of the per-shard gang-feasibility bitmasks").  The object
// that outgrows a GPU is the Q x N score matrix, so THAT is what shards: every rank holds the (small) node table, builds K1 +
// K2 for its node range only -- cut at top-level domain boundaries, so every candidate domain of a gang lies in one shard --
// and contributes one int32[G + Q] vector of per-shard feasibility counts and capacity counts; their SUM over the ranks (the
// one collective, issued by the caller on its own communicator) says which gangs cannot fit anywhere in the snapshot.
// ---------------------------------------------------------------------------------------------
int32_t grove_shard_range(grove_engine_t* e, uint32_t* lo, uint32_t* hi) {
  if (!e || !lo || !hi) return GROVE_ERR_INVALID_ARG;
  if (!e->nodes_loaded) return fail(e, GROVE_ERR_STATE, "no node snapshot loaded");
  *lo = e->shard_lo; *hi = e->shard_hi;
  return GROVE_OK;
}

int32_t grove_run_score_pass(grove_engine_t* e, float* ms) {
  if (!e) return GROVE_ERR_INVALID_ARG;
  if (ms) *ms = 0.f;
  int32_t rc = cycle_begin(e);   // allocations, derived gang tables, state resets: the pass leaves the handle ready for a cycle
  if (rc) return rc;
  CycleGuard guard{e};
  e->score_pass_valid = false; e->score_valid = false;
  if (e->G == 0 || e->Q == 0) { e->in_cycle = false; guard.armed = false; return GROVE_OK; }
  const Topo tp = make_topo(e); const Tables tb = make_tables(e); const Relax rx = make_relax(e);
  const uint32_t c0 = e->shard_lo >> 4, c1 = (e->shard_hi + 15u) >> 4, cpr = c1 > c0 ? c1 - c0 : 0u;
  const size_t tstride = size_t(cpr) << 4;
  if (e->d_T.ensure(std::max<size_t>(size_t(e->Q) * tstride, 1)) != cudaSuccess) { (void)cudaGetLastError(); return fail(e, GROVE_ERR_OOM, "score matrix shard does not fit in device memory"); }
  CU_TRY(e, cudaEventRecord(e->ev_s0, e->stream));
  rc = build_cap_tables(e, tp, tb, rx);   // K1: fit bitmap + capacities of every signature over the loaded snapshot
  if (rc) return rc;
  CU_TRY(e, e->d_F0.ensure(std::max<size_t>(size_t(e->n_sigs) * e->words, 1)));
  CU_TRY(e, cudaMemcpyAsync(e->d_F0.p, e->d_F.p, sizeof(uint32_t) * size_t(e->n_sigs) * e->words, cudaMemcpyDeviceToDevice, e->stream));
  if (cpr) k_score<<<dim3(1, std::min<uint32_t>(e->Q, 65535u)), 256, 0, e->stream>>>(tp, tb, e->d_F0.p, e->d_T.p, e->Q, c0, cpr, tstride);   // K2, this shard's columns
  CU_TRY(e, cudaGetLastError());
  CU_TRY(e, cudaEventRecord(e->ev_s1, e->stream));
  CU_TRY(e, cudaEventSynchronize(e->ev_s1));
  float t = 0; cudaEventElapsedTime(&t, e->ev_s0, e->ev_s1);
  if (ms) *ms = t;
  e->last.ms_score = t;
  e->in_cycle = false; guard.armed = false;
  e->score_pass_valid = true; e->t_c0 = c0; e->t_cpr = cpr;
  return GROVE_OK;
}

int32_t grove_shard_summary_device(grove_engine_t* e, void* d_out, uint32_t cap_words) {
  if (!e || !d_out) return GROVE_ERR_INVALID_ARG;
  if (!e->score_pass_valid) return fail(e, GROVE_ERR_STATE, "no score pass over the loaded snapshot");
  if (cap_words < e->G + e->Q) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  const Topo tp = make_topo(e); const Tables tb = make_tables(e);
  CU_TRY(e, e->d_sig_sum.ensure(std::max<uint32_t>(e->n_sigs, 1)));
  if (e->n_sigs) k_sig_range_sum<<<e->n_sigs, 256, 0, e->stream>>>(tp, e->d_cap8.p, e->shard_lo, e->shard_hi, e->d_sig_sum.p);
  k_shard_summary<<<std::max(1u, std::min((e->G * 32 + 255) / 256, e->n_sm * 8u)), 256, 0, e->stream>>>(tp, tb, e->d_cap8.p, e->d_capsum.p, e->d_sig_sum.p, e->shard_lo, e->shard_hi,
                                                                                                   static_cast<int32_t*>(d_out));
  CU_TRY(e, cudaGetLastError());
  CU_TRY(e, cudaStreamSynchronize(e->stream));   // the caller's collective runs on its own stream
  return GROVE_OK;
}

// ---- introspection for parity tests ----
int32_t grove_debug_get_perm(grove_engine_t* e, uint32_t* sorted_to_caller, uint32_t cap) {
  if (!e || !sorted_to_caller) return GROVE_ERR_INVALID_ARG;
  if (!e->nodes_loaded) return fail(e, GROVE_ERR_STATE, "no node snapshot loaded");
  if (cap < e->N) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  std::memcpy(sorted_to_caller, e->perm.data(), sizeof(uint32_t) * e->N);
  return GROVE_OK;
}

// K1 over the cycle-start snapshot is recomputed on request (the engine's own table follows the committed state)
int32_t grove_debug_get_fit_row(grove_engine_t* e, uint32_t clique, uint32_t* words, uint32_t cap_words) {
  if (!e || !words) return GROVE_ERR_INVALID_ARG;
  if (!e->have_results || clique >= e->Q) return fail(e, GROVE_ERR_STATE, "no completed cycle / bad clique");
  const uint32_t w = (e->N + 31) / 32;
  if (cap_words < w) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  { int32_t rc = grove_build_score_matrix(e, nullptr); if (rc) return rc; }
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  // the fit row of the cycle-start snapshot is the support of the score row
  std::vector<uint8_t> row(e->N);
  CU_TRY(e, cudaMemcpy(row.data(), e->d_T.p + size_t(clique) * e->Npad, e->N, cudaMemcpyDeviceToHost));
  std::memset(words, 0, sizeof(uint32_t) * w);
  for (uint32_t n = 0; n < e->N; ++n) if (row[n]) words[n >> 5] |= 1u << (n & 31);
  return GROVE_OK;
}

int32_t grove_debug_get_score_row(grove_engine_t* e, uint32_t clique, uint8_t* bytes, uint32_t cap_bytes) {
  if (!e || !bytes) return GROVE_ERR_INVALID_ARG;
  if (e->score_pass_valid) {   // after a score pass: this handle's shard of the row, zeros outside it
    if (clique >= e->Q) return fail(e, GROVE_ERR_STATE, "bad clique");
    if (cap_bytes < e->N) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
    CU_TRY(e, cudaSetDevice(e->cfg.device));
    std::memset(bytes, 0, e->N);
    const size_t first = size_t(e->t_c0) << 4, width = size_t(e->t_cpr) << 4;
    const size_t cnt = first < e->N ? std::min<size_t>(width, e->N - first) : 0;
    if (cnt) CU_TRY(e, cudaMemcpy(bytes + first, e->d_T.p + size_t(clique) * width, cnt, cudaMemcpyDeviceToHost));
    return GROVE_OK;
  }
  if (!e->have_results || clique >= e->Q) return fail(e, GROVE_ERR_STATE, "no completed cycle / bad clique");
  if (cap_bytes < e->N) return fail(e, GROVE_ERR_LIMIT, "output buffer too small");
  { int32_t rc = grove_build_score_matrix(e, nullptr); if (rc) return rc; }
  CU_TRY(e, cudaSetDevice(e->cfg.device));
  CU_TRY(e, cudaMemcpy(bytes, e->d_T.p + size_t(clique) * e->Npad, e->N, cudaMemcpyDeviceToHost));
  return GROVE_OK;
}

}  // extern "C"
