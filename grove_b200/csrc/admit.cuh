// admit.cuh -- K3: evaluation of one gang against its view of the cluster (warp-cooperative packing).
#pragma once
#include "common.cuh"

#ifdef GROVE_INLINE_ALL
#define GROVE_NI __forceinline__
#else
#define GROVE_NI __noinline__
#endif

namespace grove {
// ------------------------------------------------------------------------------------------------
// K3: gang admission.
//
// The cycle's result is the sequential pass (gangs in order rank, each against the state the earlier ones
// left).  The engine reaches it by relaxation: every gang of the window is evaluated against ITS VIEW =
// committed state minus the tentative claims of the gangs that rank before it (relax.cuh), again and again
// until nobody's view changes.  This file is one such evaluation, by ONE WARP:
//   * candidates of the gang's level are taken in score order, 32 at a time: a lane each runs the cheap
//     pre-filter on the per-signature capacity tables (a necessary condition), then the plausible ones are
//     ATTEMPTED ONE AFTER THE OTHER, IN ORDER, the first success is the answer;
//   * an attempt packs scope by scope, clique by clique, with the whole warp: lanes = the 32 nodes of a
//     fit word, capacities from the capacity bytes (nodes nobody claims) or from the node record minus
//     the claims of lower ranks minus the gang's own pods (claimed / touched nodes), prefix sums take the
//     pods in visiting order.  No per-lane stacks, no local memory.
// `extent` = how far along the gang's node visiting order this evaluation may have read node state: only a
// withdrawn claim in front of it can change the result (relax.cuh k_detect).
// ------------------------------------------------------------------------------------------------
struct GangRegs {   // per-gang constants
  uint32_t a, L, n, rank;
  uint32_t anc_lo[GROVE_MAX_LEVELS], anc_hi[GROVE_MAX_LEVELS];
};

struct GangShared {
  uint4 clq[GROVE_MAX_GANG_CLIQUES];       // req_cpu, req_mem, req_gpu, min | replicas << 8 | level << 16 | preferred << 24
  grove_scope_t scopes[GROVE_MAX_GANG_SCOPES];
  uint32_t sig[GROVE_MAX_GANG_CLIQUES];    // fit-bitmap / capacity row of each clique
  uint32_t smask[GROVE_MAX_GANG_CLIQUES];  // class mask | need_depth << 16
  uint32_t ent_node[GROVE_MAX_GANG_PODS];
  uint16_t ent_meta[GROVE_MAX_GANG_PODS];  // clique_rel
  uint32_t Hlo[GROVE_MAX_GANG_CLIQUES], Hhi[GROVE_MAX_GANG_CLIQUES];
  uint32_t s_lo[GROVE_MAX_GANG_SCOPES];
  float4 rcp[GROVE_MAX_GANG_CLIQUES];      // 1 / request per resource (0 where nothing is requested)
  int8_t c_got[GROVE_MAX_GANG_CLIQUES];    // level each clique / scope was packed at (-1: the whole cluster)
  int8_t s_got[GROVE_MAX_GANG_SCOPES];
};

// Ordered pieces of [lo,hi): descending score, ties by ascending rotated index (n - anchor) mod N.
// from == L: node granularity (ring l = anc_l \ anc_{l+1}, upper part then lower part);
// from <  L: level-`from` domain granularity (the anchor's own domain whole, then the rings).
__device__ __forceinline__ int make_pieces(const GangRegs& g, uint32_t lo, uint32_t hi, uint32_t from,
                                           uint32_t* plo, uint32_t* phi) {
  int k = 0;
  if (g.a < lo || g.a >= hi) { plo[0] = lo; phi[0] = hi; return hi > lo ? 1 : 0; }
  uint32_t prev_lo = g.a, prev_hi = g.a;
  if (from < g.L) {
    prev_lo = max(g.anc_lo[from], lo); prev_hi = min(g.anc_hi[from], hi);
    if (prev_hi > prev_lo) { plo[k] = prev_lo; phi[k] = prev_hi; ++k; }
  }
  for (int l = int(min(from, g.L)) - 1; l >= 0; --l) {
    uint32_t cl = max(g.anc_lo[l], lo), ch = min(g.anc_hi[l], hi);
    if (ch > prev_hi) { plo[k] = prev_hi; phi[k] = ch; ++k; }
    if (prev_lo > cl) { plo[k] = cl; phi[k] = prev_lo; ++k; }
    prev_lo = min(cl, prev_lo); prev_hi = max(ch, prev_hi);
  }
  if (hi > prev_hi) { plo[k] = prev_hi; phi[k] = hi; ++k; }
  if (prev_lo > lo) { plo[k] = lo; phi[k] = prev_lo; ++k; }
  return k;
}

// The same ordered pieces as make_pieces, produced one at a time from a few registers (no per-thread
// arrays: the scalar evaluator runs one attempt per LANE and every local-memory word costs a cache line
// per warp).
struct PieceIt {
  uint32_t lo, hi, prev_lo, prev_hi, first_lo, first_hi;
  int l, stage;  // stage: 0 first piece pending, 1 rings (upper), 2 rings (lower), 3 tail upper, 4 tail lower, 5 done
  bool outside;
  __device__ __forceinline__ void init(const GangRegs& g, uint32_t lo_, uint32_t hi_, uint32_t from) {
    lo = lo_; hi = hi_;
    outside = g.a < lo || g.a >= hi;
    stage = 0; prev_lo = g.a; prev_hi = g.a; first_lo = first_hi = 0;
    l = int(min(from, g.L)) - 1;
    if (!outside && from < g.L) {
      first_lo = max(g.anc_lo[from], lo); first_hi = min(g.anc_hi[from], hi);
      prev_lo = first_lo; prev_hi = first_hi;
    }
  }
  __device__ __forceinline__ bool next(const GangRegs& g, uint32_t& a, uint32_t& b) {
    if (outside) { if (stage == 0 && hi > lo) { stage = 5; a = lo; b = hi; return true; } return false; }
    if (stage == 0) { stage = 1; if (first_hi > first_lo) { a = first_lo; b = first_hi; return true; } }
    while (stage == 1 || stage == 2) {
      if (l < 0) { stage = 3; break; }
      const uint32_t cl = max(g.anc_lo[l], lo), ch = min(g.anc_hi[l], hi);
      if (stage == 1) { stage = 2; if (ch > prev_hi) { a = prev_hi; b = ch; return true; } }
      // stage 2: lower part of ring l, then move one level out
      const uint32_t pl = prev_lo;
      prev_lo = min(cl, prev_lo); prev_hi = max(ch, prev_hi);
      --l; stage = 1;
      if (pl > cl) { a = cl; b = pl; return true; }
    }
    if (stage == 3) { stage = 4; if (hi > prev_hi) { a = prev_hi; b = hi; return true; } }
    if (stage == 4) { stage = 5; if (prev_lo > lo) { a = lo; b = prev_lo; return true; } }
    return false;
  }
};

__device__ __forceinline__ uint32_t cap_from(uint32_t cpu, uint32_t mem, uint32_t gpu, uint32_t pods, const uint4& q) {
  uint32_t c = pods;
  if (q.x) c = min(c, div_small(cpu, q.x));
  if (q.y) c = min(c, div_small(mem, q.y));
  if (q.z) c = min(c, div_small(gpu, q.z));
  return c;
}

// floor(x / d) for the staged evaluator, exact below 256 and >= 256 above (callers never ask for more than 255 pods);
// r = 1.0f / d.  Branch-free so that the three resources -- and the nodes a lane handles -- overlap: the estimate is
// within one of the quotient (relative error of the product < 2^-22, quotients < 257), one signed remainder fixes it.
__device__ __forceinline__ uint32_t div_rcp(uint32_t x, uint32_t d, float r) {
  uint32_t q = __float2uint_rz(fminf(__uint2float_rz(x) * r, 256.0f));
  const long long rem = (long long)x - (long long)((unsigned long long)q * d);
  q += uint32_t(rem >= (long long)d) - uint32_t(rem < 0);
  return d ? q : 0xFFFFu;
}
__device__ __forceinline__ uint32_t cap_from_rcp(uint32_t cpu, uint32_t mem, uint32_t gpu, uint32_t pods, const uint4& q, const float4& r) {
  return min(min(div_rcp(cpu, q.x, r.x), div_rcp(mem, q.y, r.y)), min(div_rcp(gpu, q.z, r.z), pods));
}

// position of node n in the gang's node visiting order (descending closeness to the anchor, ties by ascending
// rotated index): the anchor's deepest domain from the anchor upwards, then its lower part, then ring by ring
__device__ __forceinline__ uint32_t visit_pos(const GangRegs& g, uint32_t n) {
  uint32_t in_lo = g.a, in_hi = g.a;   // the domain one level deeper than the ring n lies in (empty below the deepest level)
  for (int l = int(g.L) - 1; l >= -1; --l) {
    const uint32_t lo = l >= 0 ? g.anc_lo[l] : 0u, hi = l >= 0 ? g.anc_hi[l] : g.n;
    if (n >= lo && n < hi && hi > lo) {
      const uint32_t inner = in_hi - in_lo;
      if (n >= in_hi) return inner + (n - in_hi);
      return inner + (hi - in_hi) + (n - lo);
    }
    if (hi > lo) { in_lo = min(in_lo, lo); in_hi = max(in_hi, hi); }
  }
  return g.n;
}

// ---- the evaluator: the whole warp packs ONE candidate range ------------------------------------------
template <bool kPref_>
struct Ev {
  static constexpr bool kPref = kPref_;
  static constexpr bool kStaged = false;
  const Topo& tp; const Relax& rb; GangShared& sh; const GangRegs& g; uint32_t lane;
  uint32_t np;
  uint32_t tmask = 0;   // bit (n & 31) set for every node the gang has put a pod on: quick 'untouched' test
  uint32_t ext = 0;     // see the file comment
  uint32_t t_stage = 0, t_pre = 0, t_pack = 0, n_stage = 0;
  __device__ Ev(const Topo& t, const Relax& r, GangShared& s, const GangRegs& gr, uint32_t ln)
      : tp(t), rb(r), sh(s), g(gr), lane(ln), np(0) {}

  // pods of clique cr that still fit on node n under the gang's view, after what the gang itself put there
  __device__ __forceinline__ uint32_t cap_view(uint32_t cr, uint32_t n) const {
    const uint32_t live = (__ldg(rb.nlive + (n >> 2)) >> ((n & 3u) * 8u)) & 0xFFu;
    const bool own = (tmask >> (n & 31u)) & 1u;
    if (!live && !own) {
      const uint32_t c = __ldg(rb.cap8 + size_t(sh.sig[cr]) * tp.npad + n);
      if (c != 255u) return c;   // nobody claims the node and the table is current: the byte is the answer
    }
    const uint4 r = __ldg(tp.nres + n);
    const uint32_t sm = sh.smask[cr];
    if (!(r.w & GROVE_NODE_SCHEDULABLE) || !((sm >> ((r.w >> GROVE_NODE_CLASS_SHIFT) & 0xFu)) & 1u) || ((r.w >> 16) & 0xFu) < (sm >> 16)) return 0u;
    int cpu = int(r.x), mem = int(r.y), gpu = int(r.z & 0xFFFFu), pods = int(r.z >> 16);
    if (live & 0x7Fu) {   // claims: all of them, minus those of the gangs that rank after this one (see EvS::begin)
      const int4 t = __ldg(rb.ctot + n);
      cpu -= t.x; mem -= t.y; gpu -= t.z; pods -= t.w;
      if (__ldg(rb.cmaxr + n) >= g.rank) {
        if (live & 0x3Fu) {
          const uint4* line = rb.claims + size_t(n) * kClaimSlots;
#pragma unroll
          for (uint32_t s = 0; s < kClaimSlots; ++s) {
            const uint4 c = __ldg(line + s);
            if (c.x >= g.rank && c.x != kClaimEmpty) { cpu += int(c.y); mem += int(c.z); gpu += int(c.w & 0xFFFFu); pods += int(c.w >> 16); }
          }
        }
        if (live & kHasOvf) {
          for (uint32_t i = __ldg(rb.ovf_head + n); i; i = __ldg(rb.ovf_next + i - 1)) {
            const uint4 c = __ldg(rb.ovf_claim + i - 1);
            if (c.x >= g.rank && c.x != kClaimEmpty) { cpu += int(c.y); mem += int(c.z); gpu += int(c.w & 0xFFFFu); pods += int(c.w >> 16); }
          }
        }
      }
    }
    if (own) {
      for (uint32_t i = 0; i < np; ++i) {
        if (sh.ent_node[i] == n) {
          const uint4 o = sh.clq[sh.ent_meta[i]];
          cpu -= int(o.x); mem -= int(o.y); gpu -= int(o.z); pods -= 1;
        }
      }
    }
    return cap_from(uint32_t(max(cpu, 0)), uint32_t(max(mem, 0)), uint32_t(max(gpu, 0)), uint32_t(max(pods, 0)), sh.clq[cr]);
  }

  __device__ __forceinline__ uint32_t scope_filter(const grove_scope_t&, uint32_t, uint32_t, bool, int) { return kFull; }   // staged evaluator only
  __device__ __forceinline__ void note_read(uint32_t last) { ext = max(ext, visit_pos(g, last) + 1u); }
  __device__ __forceinline__ void begin(uint32_t, uint32_t) { np = 0; tmask = 0; }       // a fresh attempt
  __device__ __forceinline__ void rollback(uint32_t mark) { np = mark; }               // drop the pods placed after mark

  // up to `want` pods of clique cr on fit nodes of [lo,hi) in score order; returns pods placed
  __device__ GROVE_NI uint32_t take(uint32_t cr, uint32_t lo, uint32_t hi, uint32_t want) {
    if (want == 0 || hi <= lo) return 0;
    const uint32_t* Frow = rb.F + size_t(sh.sig[cr]) * tp.words;
    PieceIt pit; pit.init(g, lo, hi, g.L);
    uint32_t placed = 0, last = GROVE_NONE_U32;
    for (uint32_t a, b; placed < want && pit.next(g, a, b);) {
      for (uint32_t base = a & ~31u; base < b && placed < want; base += 32) {
        uint32_t word = __ldg(Frow + (base >> 5));
        if (base < a) word &= kFull << (a - base);
        if (base + 32u > b) word &= (1u << (b - base)) - 1u;
        last = min(base + 31u, b - 1u);
        if (!word) continue;   // no fit node when the tables were built: none now
        const uint32_t n = base + lane;
        const uint32_t c = ((word >> lane) & 1u) ? cap_view(cr, n) : 0u;
        const uint32_t incl = warp_incl_scan(c, lane), excl = incl - c, rem = want - placed;
        const uint32_t t = excl >= rem ? 0u : min(c, rem - excl);
        const uint32_t tincl = warp_incl_scan(t, lane);
        __syncwarp();  // every lane's scan of the entry stack is over before it grows
        if (t) {
          const uint32_t pos = np + tincl - t;
          for (uint32_t j = 0; j < t; ++j) { sh.ent_node[pos + j] = n; sh.ent_meta[pos + j] = uint16_t(cr); }
        }
        const uint32_t tb = __ballot_sync(kFull, t != 0);
        const uint32_t tot = __shfl_sync(kFull, tincl, 31);
        tmask |= tb;   // base is 32-aligned: lane == n & 31
        np += tot; placed += tot;
        if (placed >= want && tb) last = base + (31u - __clz(tb));
        __syncwarp();
      }
    }
    if (last != GROVE_NONE_U32) note_read(last);
    return placed;
  }

  __device__ bool fill_min(uint32_t cr, uint32_t lo, uint32_t hi) {
    const uint32_t m = sh.clq[cr].w & 0xFFu;
    const uint32_t mark = np;
    if (take(cr, lo, hi, m) < m) { rollback(mark); return false; }
    if (lane == 0) { sh.Hlo[cr] = lo; sh.Hhi[cr] = hi; }
    __syncwarp();
    return true;
  }

  // clique whose own Required level is a unit level (one node per domain, e.g. hostname):
  // first node of [lo,hi) in score order that takes all m pods
  __device__ GROVE_NI bool find_unit(uint32_t cr, uint32_t lo, uint32_t hi) {
    const uint32_t m = sh.clq[cr].w & 0xFFu;
    const uint32_t* Frow = rb.F + size_t(sh.sig[cr]) * tp.words;
    PieceIt pit; pit.init(g, lo, hi, g.L);
    uint32_t last = GROVE_NONE_U32;
    for (uint32_t a, b; pit.next(g, a, b);) {
      for (uint32_t base = a & ~31u; base < b; base += 32) {
        uint32_t word = __ldg(Frow + (base >> 5));
        if (base < a) word &= kFull << (a - base);
        if (base + 32u > b) word &= (1u << (b - base)) - 1u;
        last = min(base + 31u, b - 1u);
        if (!word) continue;
        const uint32_t n = base + lane;
        const uint32_t c = ((word >> lane) & 1u) ? cap_view(cr, n) : 0u;
        const uint32_t okb = __ballot_sync(kFull, c >= m && ((word >> lane) & 1u));
        __syncwarp();
        if (okb) {
          const uint32_t nn = base + (__ffs(okb) - 1);
          for (uint32_t j = lane; j < m; j += 32) { sh.ent_node[np + j] = nn; sh.ent_meta[np + j] = uint16_t(cr); }
          if (lane == 0) { sh.Hlo[cr] = nn; sh.Hhi[cr] = nn + 1; }
          tmask |= 1u << (nn & 31u);
          np += m;
          note_read(nn);
          __syncwarp();
          return true;
        }
      }
    }
    if (last != GROVE_NONE_U32) note_read(last);
    return false;
  }
};


// ---- staged evaluator: the candidate range lives in shared memory -------------------------------------------
// For a candidate of at most kStageMax nodes (a rack, a block) the warp first computes the gang's VIEW of every node
// of the range -- committed state minus the claims of lower ranks -- into shared memory (two rounds of independent
// loads), then packs from there: capacities are divisions on the staged record, pods the gang places are subtracted
// from it in place (no entry-stack scans), a failed scope adds them back.  An attempt costs a few thousand cycles
// instead of a chain of dependent L2 look-ups per 32 nodes.
constexpr uint32_t kStageMax = 128;

template <bool kPref_>
struct EvS {
  static constexpr bool kPref = kPref_;
  static constexpr bool kStaged = true;   // node state in shared memory: an attempt costs less than the table look-ups that would skip it
  const Topo& tp; const Relax& rb; GangShared& sh; const GangRegs& g; uint32_t lane;
  int4* view;           // [kStageMax] cpu, mem, gpu, pods the gang may still take.  Signed: the claims of lower ranks may transiently exceed
                        // the committed state (saturating subtraction claim by claim == clamping the sum at zero when it is read)
  uint32_t* vflag;      // [kStageMax] node flags | vdepth << 16
  uint8_t* rk;          // [kStageMax + 256] sub-domain filter scratch: the sub-domain (lane) each staged node belongs to, then
                        // per-sub-domain sum and max (32 words each) of the pods of ONE clique that fit
  uint32_t t_stage = 0, t_pre = 0, t_pack = 0, n_stage = 0;   // GROVE_DEBUG_ADMIT: cycles staging / pre-filtering sub-domains / packing
  uint32_t t_st2 = 0, t_st3 = 0;                              // of the staging: claim lines, overflow chains
  uint32_t vlo = 0, vhi = 0;
  uint32_t np;
  uint32_t tmask = 0;
  uint32_t ext = 0;
  __device__ EvS(const Topo& t, const Relax& r, GangShared& s, const GangRegs& gr, uint32_t ln, int4* v, uint32_t* vf, uint8_t* cv)
      : tp(t), rb(r), sh(s), g(gr), lane(ln), view(v), vflag(vf), rk(cv), np(0) {}

  // Stage the gang's view of [dl, dh): committed record minus the claims of the ranks before it.  A lane per node, four nodes a
  // lane, ONE L2 round trip for almost every node: the record, the node's claim TOTAL (all ranks) and the highest rank that ever
  // claimed it (relax.cuh ctot / cmaxr).  Gangs enter the window in rank order, so for most evaluations every claim on a node is
  // of a lower rank and the view is record - total.  Only where a HIGHER rank may lean on the node (cmaxr >= rank) are its claim
  // line and overflow chain read, to give those claims back.
  __device__ GROVE_NI void begin(uint32_t dl, uint32_t dh) {
    np = 0; vlo = dl; vhi = dh;
    const long long tb0 = rb.dbg ? clock64() : 0;
    __syncwarp();
    constexpr uint32_t kPer = kStageMax / 32;
    uint4 r[kPer]; int4 t[kPer]; uint32_t live[kPer], mr[kPer];
#pragma unroll
    for (uint32_t k = 0; k < kPer; ++k) {
      const uint32_t n = dl + k * 32u + lane;
      const bool in = n < dh;
      r[k] = in ? __ldg(tp.nres + n) : make_uint4(0, 0, 0, 0);
      t[k] = in ? __ldg(rb.ctot + n) : make_int4(0, 0, 0, 0);
      mr[k] = in ? __ldg(rb.cmaxr + n) : 0u;
      live[k] = in ? (__ldg(rb.nlive + (n >> 2)) >> ((n & 3u) * 8u)) & 0x7Fu : 0u;
    }
    const long long tc0 = rb.dbg ? clock64() : 0;
#pragma unroll
    for (uint32_t k = 0; k < kPer; ++k) {
      const uint32_t n = dl + k * 32u + lane;
      int cpu = int(r[k].x) - t[k].x, mem = int(r[k].y) - t[k].y, gpu = int(r[k].z & 0xFFFFu) - t[k].z, pods = int(r[k].z >> 16) - t[k].w;
      if (live[k] && mr[k] >= g.rank) {   // a gang of a higher rank may hold a claim here: it is invisible to this one
        if (live[k] & 0x3Fu) {
          const uint4* line = rb.claims + size_t(n) * kClaimSlots;
          uint4 c[kClaimSlots];
#pragma unroll
          for (uint32_t s = 0; s < kClaimSlots; ++s) c[s] = __ldg(line + s);
#pragma unroll
          for (uint32_t s = 0; s < kClaimSlots; ++s)
            if (c[s].x >= g.rank && c[s].x != kClaimEmpty) { cpu += int(c[s].y); mem += int(c[s].z); gpu += int(c[s].w & 0xFFFFu); pods += int(c[s].w >> 16); }
        }
        if (live[k] & kHasOvf) {
          for (uint32_t i = __ldg(rb.ovf_head + n); i; i = __ldg(rb.ovf_next + i - 1)) {
            const uint4 c = __ldg(rb.ovf_claim + i - 1);
            if (c.x >= g.rank && c.x != kClaimEmpty) { cpu += int(c.y); mem += int(c.z); gpu += int(c.w & 0xFFFFu); pods += int(c.w >> 16); }
          }
        }
      }
      view[k * 32u + lane] = make_int4(cpu, mem, gpu, pods);
      vflag[k * 32u + lane] = r[k].w;
    }
    __syncwarp();
    // the whole range has been read: it ends at the furthest position any of its nodes has in the visiting order
    ext = max(ext, (g.a >= dl && g.a < dh) ? dh - dl : visit_pos(g, dh - 1u) + 1u);
    if (rb.dbg) { const long long te = clock64(); t_stage += uint32_t(te - tb0); t_st2 += uint32_t(tc0 - tb0); t_st3 += uint32_t(te - tc0); ++n_stage; }
  }

  __device__ __forceinline__ uint32_t cap(uint32_t cr, uint32_t n) const {
    const int4 v = view[n - vlo];
    const uint32_t f = vflag[n - vlo];
    const uint32_t sm = sh.smask[cr];
    const bool usable = (f & GROVE_NODE_SCHEDULABLE) && ((sm >> ((f >> GROVE_NODE_CLASS_SHIFT) & 0xFu)) & 1u) && ((f >> 16) & 0xFu) >= (sm >> 16);
    const uint32_t c = cap_from_rcp(uint32_t(max(v.x, 0)), uint32_t(max(v.y, 0)), uint32_t(max(v.z, 0)), uint32_t(max(v.w, 0)), sh.clq[cr], sh.rcp[cr]);
    return usable ? c : 0u;
  }

  // Sub-domain filter on the staged view: which of the (at most 32) level-sl domains [el, eh) -- a lane each -- could take
  // every clique of scope s on its own?  A necessary condition like the table look-ups of scope_plausible, but against what
  // the gang really sees (the tables only know the committed state as of their last build): a candidate whose racks are
  // taken by lower ranks' claims fails here instead of after an attempt per rack.
  __device__ GROVE_NI uint32_t scope_filter(const grove_scope_t& s, uint32_t el, uint32_t eh, bool in, int sl) {
    constexpr uint32_t kPer = kStageMax / 32;
    uint32_t* rsum = reinterpret_cast<uint32_t*>(rk + kStageMax);
    uint32_t* rmax = rsum + 32;
    bool ok = in;
    el = max(el, vlo); eh = min(eh, vhi);
    __syncwarp();
    reinterpret_cast<uint32_t*>(rk)[lane] = kFull;             // a node that lacks the label is in no sub-domain
    __syncwarp();
    if (in) for (uint32_t n = el; n < eh; ++n) rk[n - vlo] = uint8_t(lane);   // (stores: nothing waits on them)
    for (uint32_t i = 0; i < s.n_cliques; ++i) {
      const uint32_t cr = s.first_clique + i;
      const uint32_t w = sh.clq[cr].w;
      const uint32_t m = w & 0xFFu, ql = (w >> 16) & 0xFFu;
      if (m == 0) continue;
      rsum[lane] = 0; rmax[lane] = 0;
      __syncwarp();
#pragma unroll
      for (uint32_t k = 0; k < kPer; ++k) {
        const uint32_t idx = k * 32u + lane;
        const uint32_t c = vlo + idx < vhi ? cap(cr, vlo + idx) : 0u;
        const uint32_t slot = rk[idx];
        if (c && slot != 0xFFu) { atomicAdd(rsum + slot, c); atomicMax(rmax + slot, c); }
      }
      __syncwarp();
      const bool one_node = ql != GROVE_LEVEL_NONE && int(ql) > sl && tp.unit[ql];   // all m pods on one node
      ok = ok && (one_node ? rmax[lane] >= m : rsum[lane] >= m);
      __syncwarp();
    }
    return __ballot_sync(kFull, ok);
  }

  // give back the pods placed after mark
  __device__ GROVE_NI void rollback(uint32_t mark) {
    __syncwarp();
    for (uint32_t i = mark + lane; i < np; i += 32) {
      const uint4 q = sh.clq[sh.ent_meta[i]];
      int* v = reinterpret_cast<int*>(view + (sh.ent_node[i] - vlo));
      if (q.x) atomicAdd(v + 0, int(q.x));
      if (q.y) atomicAdd(v + 1, int(q.y));
      if (q.z) atomicAdd(v + 2, int(q.z));
      atomicAdd(v + 3, 1);
    }
    np = mark;
    __syncwarp();
  }

  __device__ GROVE_NI uint32_t take(uint32_t cr, uint32_t lo, uint32_t hi, uint32_t want) {
    if (want == 0 || hi <= lo) return 0;
    const uint4 q = sh.clq[cr];
    PieceIt pit; pit.init(g, lo, hi, g.L);
    uint32_t placed = 0;
    for (uint32_t a, b; placed < want && pit.next(g, a, b);) {
      for (uint32_t base = a & ~31u; base < b && placed < want; base += 32) {
        const uint32_t n = base + lane;
        const uint32_t c = (n >= a && n < b) ? cap(cr, n) : 0u;
        if (!__any_sync(kFull, c != 0u)) continue;
        const uint32_t incl = warp_incl_scan(c, lane), excl = incl - c, rem = want - placed;
        const uint32_t t = excl >= rem ? 0u : min(c, rem - excl);
        const uint32_t tincl = warp_incl_scan(t, lane);
        if (t) {
          const uint32_t pos = np + tincl - t;
          for (uint32_t j = 0; j < t; ++j) { sh.ent_node[pos + j] = n; sh.ent_meta[pos + j] = uint16_t(cr); }
          int4 v = view[n - vlo];
          v.x -= int(t * q.x); v.y -= int(t * q.y); v.z -= int(t * q.z); v.w -= int(t);
          view[n - vlo] = v;
        }
        const uint32_t tot = __shfl_sync(kFull, tincl, 31);
        np += tot; placed += tot;
        __syncwarp();
      }
    }
    return placed;
  }

  __device__ bool fill_min(uint32_t cr, uint32_t lo, uint32_t hi) {
    const uint32_t m = sh.clq[cr].w & 0xFFu;
    const uint32_t mark = np;
    if (take(cr, lo, hi, m) < m) { rollback(mark); return false; }
    if (lane == 0) { sh.Hlo[cr] = lo; sh.Hhi[cr] = hi; }
    __syncwarp();
    return true;
  }

  __device__ GROVE_NI bool find_unit(uint32_t cr, uint32_t lo, uint32_t hi) {
    const uint32_t m = sh.clq[cr].w & 0xFFu;
    const uint4 q = sh.clq[cr];
    PieceIt pit; pit.init(g, lo, hi, g.L);
    for (uint32_t a, b; pit.next(g, a, b);) {
      for (uint32_t base = a & ~31u; base < b; base += 32) {
        const uint32_t n = base + lane;
        const bool in = n >= a && n < b;
        const uint32_t c = in ? cap(cr, n) : 0u;
        const uint32_t okb = __ballot_sync(kFull, in && c >= m);
        if (okb) {
          const uint32_t nn = base + (__ffs(okb) - 1);
          for (uint32_t j = lane; j < m; j += 32) { sh.ent_node[np + j] = nn; sh.ent_meta[np + j] = uint16_t(cr); }
          if (lane == 0) {
            sh.Hlo[cr] = nn; sh.Hhi[cr] = nn + 1;
            int4 v = view[nn - vlo];
            v.x -= int(m * q.x); v.y -= int(m * q.y); v.z -= int(m * q.z); v.w -= int(m);
            view[nn - vlo] = v;
          }
          np += m;
          __syncwarp();
          return true;
        }
      }
    }
    return false;
  }
};

// ---- candidate pre-filter: a NECESSARY condition for place_in(lo, hi) to succeed ------------------
// (each clique alone must find MinReplicas worth of capacity in a domain it could be packed into, and
// the cliques of a scope must find it inside one common scope domain).  Reads only the small
// per-signature capacity tables.
__device__ __forceinline__ bool clique_plausible(const Topo& tp, const Relax& rb, const GangShared& sh, uint32_t cr,
                                 uint32_t lo, uint32_t hi, int lvl, uint32_t dE) {
  const uint32_t w = sh.clq[cr].w;
  const uint32_t m = w & 0xFFu, ql = (w >> 16) & 0xFFu;
  if (m == 0) return true;
  const size_t row = size_t(sh.sig[cr]);
  const bool tabled = lvl >= 0 && !tp.unit[lvl];
  if (ql != GROVE_LEVEL_NONE && int(ql) > lvl) {
    if (tp.unit[ql]) {  // all m pods on one node
      if (tabled) return __ldg(rb.capmax + row * tp.cap_stride + tp.cap_off[lvl] + dE) >= m;
      for (uint32_t n = lo; n < hi; ++n) if (__ldg(rb.cap8 + row * tp.npad + n) >= m) return true;
      return false;
    }
    const uint32_t d0 = __ldg(tp.next_dom[ql] + lo), d1 = __ldg(tp.next_dom[ql] + hi);
    uint32_t any = 0;  // no early exit: the look-ups are independent and overlap
    for (uint32_t d = d0; d < d1; ++d) any |= __ldg(rb.capsum + row * tp.cap_stride + tp.cap_off[ql] + d) >= m;
    return any != 0;
  }
  if (tabled) return __ldg(rb.capsum + row * tp.cap_stride + tp.cap_off[lvl] + dE) >= m;
  uint32_t sum = 0;
  for (uint32_t n = lo; n < hi && sum < m; ++n) sum += __ldg(rb.cap8 + row * tp.npad + n);
  return sum >= m;
}

__device__ __forceinline__ bool scope_plausible(const Topo& tp, const Relax& rb, const GangShared& sh, const grove_scope_t& s,
                                uint32_t lo, uint32_t hi, int lvl, uint32_t dE) {
  uint32_t all = 1;
  for (uint32_t i = 0; i < s.n_cliques; ++i) all &= clique_plausible(tp, rb, sh, s.first_clique + i, lo, hi, lvl, dE);
  return all != 0;
}

// one scope of a gang inside the candidate [lo, hi) of level lvl
__device__ __forceinline__ bool scope_ok(const Topo& tp, const Relax& rb, const GangShared& sh, const grove_scope_t& s,
                                         uint32_t lo, uint32_t hi, int lvl, uint32_t dD) {
  if (s.level != GROVE_LEVEL_NONE && int(s.level) > lvl) {
    const uint32_t d0 = __ldg(tp.next_dom[s.level] + lo), d1 = __ldg(tp.next_dom[s.level] + hi);
    uint32_t any = 0;  // no early exit: children are independent table look-ups
    for (uint32_t d = d0; d < d1; ++d)
      any |= scope_plausible(tp, rb, sh, s, __ldg(tp.dom_lo[s.level] + d), __ldg(tp.dom_hi[s.level] + d), int(s.level), d);
    return any != 0;
  }
  return scope_plausible(tp, rb, sh, s, lo, hi, lvl, dD);
}

__device__ bool gang_plausible(const Topo& tp, const Relax& rb, const GangShared& sh, uint32_t n_scopes,
                               uint32_t lo, uint32_t hi, int lvl, uint32_t dD) {
  for (uint32_t si = 0; si < n_scopes; ++si)
    if (!scope_ok(tp, rb, sh, sh.scopes[si], lo, hi, lvl, dD)) return false;
  return true;
}

// Levels a unit (gang / scope / clique) with constraint (req, pref) is tried at inside a parent range of
// level lvl (-1 = whole cluster): `first` down to the returned base.  base = the hard level (Required when
// deeper than the parent's, else the parent range itself); a deeper Preferred level is tried first and
// widened level by level up to base (podgang.go:110-117).  Oracle: level_span().  kPref = false: the submission
// carries no Preferred level anywhere, the walk is the single step `base` (the kernels are instantiated both ways so
// that Required-only workloads run the loop-free code).
template <bool kPref>
__device__ __forceinline__ int level_span(uint32_t req, uint32_t pref, int lvl, int& first) {
  const int base = (req != GROVE_LEVEL_NONE && int(req) > lvl) ? int(req) : lvl;
  first = (kPref && pref != GROVE_LEVEL_NONE && int(pref) > base) ? int(pref) : base;
  return base;
}

template <class Ev>
__device__ GROVE_NI bool place_scope(Ev& ev, const grove_scope_t& s, uint32_t lo, uint32_t hi, int lvl) {
  const Topo& tp = ev.tp;
  const uint32_t mark = ev.np;
  for (uint32_t i = 0; i < s.n_cliques; ++i) {
    const uint32_t cr = s.first_clique + i;
    const uint32_t w = ev.sh.clq[cr].w;
    const uint32_t m = w & 0xFFu;
    bool ok = false;
    int first;
    const int base = level_span<Ev::kPref>((w >> 16) & 0xFFu, w >> 24, lvl, first);
    int ql = first;
    do {
      if (ql > lvl) {
        // find_unit scans fit NODES: every fit node is a domain of a Required unit level (the fit row demands the
        // labels down to it), but not of a Preferred one (ragged labels) -- those take the domain walk below
        if (tp.unit[ql] && m >= 1 && ql == base) {
          ok = ev.find_unit(cr, lo, hi);
        } else {
          PieceIt pit; pit.init(ev.g, lo, hi, uint32_t(ql));
          for (uint32_t pa, pb; !ok && pit.next(ev.g, pa, pb);) {
            const uint32_t d0 = __ldg(tp.next_dom[ql] + pa), d1 = __ldg(tp.next_dom[ql] + pb);
            for (uint32_t d = d0; d < d1 && !ok; ++d)
              ok = ev.fill_min(cr, __ldg(tp.dom_lo[ql] + d), __ldg(tp.dom_hi[ql] + d));
          }
        }
      } else {
        ok = ev.fill_min(cr, lo, hi);
      }
      if (ok && ev.lane == 0) ev.sh.c_got[cr] = int8_t(ql);
    } while (Ev::kPref && !ok && --ql >= base);
    if (!ok) { ev.rollback(mark); return false; }
  }
  return true;
}

template <class Ev>
__device__ GROVE_NI bool place_in(Ev& ev, uint32_t n_scopes, uint32_t lo, uint32_t hi, int lvl) {
  const Topo& tp = ev.tp;
  // (staged evaluator) the first / end domain index of every deeper level inside [lo, hi): asked for BEFORE the staging so that
  // the look-ups overlap it -- each scope with a narrower level would otherwise start with one more L2 round trip
  uint32_t pd0[GROVE_MAX_LEVELS], pd1[GROVE_MAX_LEVELS];
#pragma unroll
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) {
    pd0[l] = pd1[l] = 0;
    if (Ev::kStaged && int(l) > lvl && l < tp.L) { pd0[l] = __ldg(tp.next_dom[l] + lo); pd1[l] = __ldg(tp.next_dom[l] + hi); }
  }
  ev.begin(lo, hi);
  for (uint32_t si = 0; si < n_scopes; ++si) {
    const grove_scope_t s = ev.sh.scopes[si];
    bool ok = false;
    int first;
    const int base = level_span<Ev::kPref>(s.level, s.preferred1 ? uint32_t(s.preferred1) - 1u : uint32_t(GROVE_LEVEL_NONE), lvl, first);
    int sl = first;
    do {
      bool filtered = false;
      if constexpr (Ev::kStaged) {
        if (sl > lvl) {
          // the staged range holds at most kStageMax nodes: usually all its level-sl domains fit one warp pass.  A lane each:
          // filter them ONCE against the staged view, then attempt the survivors in visiting order (piece by piece, ascending
          // inside a piece -- the order of the general walk below)
          uint32_t d0 = 0, d1 = 0;
#pragma unroll
          for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) if (int(l) == sl) { d0 = pd0[l]; d1 = pd1[l]; }
          if (d1 - d0 <= 32u) {
            filtered = true;
            const long long tp0 = ev.rb.dbg ? clock64() : 0;
            const bool in = d0 + ev.lane < d1;
            uint32_t el = 0, eh = 0;
            if (in) { el = __ldg(tp.dom_lo[sl] + d0 + ev.lane); eh = __ldg(tp.dom_hi[sl] + d0 + ev.lane); }
            const uint32_t plaus = ev.scope_filter(s, el, eh, in, sl);
            const long long tp1 = ev.rb.dbg ? clock64() : 0;
            PieceIt pit; pit.init(ev.g, lo, hi, uint32_t(sl));
            for (uint32_t pa, pb; !ok && plaus && pit.next(ev.g, pa, pb);) {
              uint32_t todo = plaus & __ballot_sync(kFull, in && el >= pa && el < pb);
              while (todo && !ok) {
                const uint32_t src = __ffs(todo) - 1; todo &= todo - 1;
                const uint32_t l0 = __shfl_sync(kFull, el, src), h0 = __shfl_sync(kFull, eh, src);
                ok = place_scope(ev, s, l0, h0, sl);
                if (ok && ev.lane == 0) ev.sh.s_lo[si] = l0;
              }
            }
            if (ev.rb.dbg) { ev.t_pre += uint32_t(tp1 - tp0); ev.t_pack += uint32_t(clock64() - tp1); }
          }
        }
      }
      if (filtered) {
      } else if (sl > lvl) {
        PieceIt pit; pit.init(ev.g, lo, hi, uint32_t(sl));
        for (uint32_t pa, pb; !ok && pit.next(ev.g, pa, pb);) {
          const uint32_t d0 = __ldg(tp.next_dom[sl] + pa), d1 = __ldg(tp.next_dom[sl] + pb);
          // 32 scope domains at a time: a lane each runs the pre-filter (the table-time capacities are an upper
          // bound: a domain that lacks them cannot be packed), the plausible ones are attempted in order
          for (uint32_t db = d0; db < d1 && !ok; db += 32) {
            const uint32_t d = db + ev.lane;
            uint32_t el = 0, eh = 0;
            bool plaus = false;
            const long long tp0 = ev.rb.dbg ? clock64() : 0;
            if (d < d1) {
              el = __ldg(tp.dom_lo[sl] + d); eh = __ldg(tp.dom_hi[sl] + d);
              plaus = scope_plausible(tp, ev.rb, ev.sh, s, el, eh, sl, d);
            }
            uint32_t todo = __ballot_sync(kFull, plaus);
            const long long tp1 = ev.rb.dbg ? clock64() : 0;
            while (todo && !ok) {
              const uint32_t src = __ffs(todo) - 1; todo &= todo - 1;
              const uint32_t l0 = __shfl_sync(kFull, el, src), h0 = __shfl_sync(kFull, eh, src);
              ok = place_scope(ev, s, l0, h0, sl);
              if (ok && ev.lane == 0) ev.sh.s_lo[si] = l0;
            }
            if (ev.rb.dbg) { ev.t_pre += uint32_t(tp1 - tp0); ev.t_pack += uint32_t(clock64() - tp1); }
          }
        }
      } else {
        ok = place_scope(ev, s, lo, hi, lvl);
        if (ok && ev.lane == 0) ev.sh.s_lo[si] = lo;
      }
      if (ok && ev.lane == 0) ev.sh.s_got[si] = int8_t(sl);
    } while (Ev::kPref && !ok && --sl >= base);
    if (!ok) { ev.np = 0; return false; }
  }
  return true;
}

// PlacementScore bookkeeping (oracle: score_unit): a unit that carries a pack constraint asked for `want` = Preferred
// if set else Required and was packed at level `got` (-1: no domain of its own): credit min(got, want) + 1 of want + 1
__device__ __forceinline__ void score_unit(uint32_t req, uint32_t pref, int got, uint32_t& num, uint32_t& den) {
  if (req == GROVE_LEVEL_NONE && pref == GROVE_LEVEL_NONE) return;
  const int want = pref != GROVE_LEVEL_NONE ? int(pref) : int(req);
  den += uint32_t(want) + 1u;
  num += uint32_t(min(got, want) + 1);
}

// The candidate pre-filter per (gang shape, domain): a CTA per 32 domains of one level, FOUR threads per domain (they share the
// gang's scopes: a base gang's scopes are independent chains of table look-ups), the shape's representative gang staged in
// shared memory.  Runs after every capacity-table build; k_eval then reads one bit per candidate.
__global__ void __launch_bounds__(128) k_shape_plaus(Topo tp, Tables tb, Relax rx, const uint32_t* __restrict__ shape_rep) {
  __shared__ GangShared sh;
  __shared__ uint32_t s_bits;
  const uint32_t shape = blockIdx.y, l = blockIdx.z;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, slot = threadIdx.x & 3u;
  pdl_begin();
  const uint32_t gi = shape_rep[shape];
  const grove_gang_t gg = tb.gangs[gi];
  // candidate levels of the shape: Preferred (if any) down to Required; the whole cluster needs no table
  int first;
  const int base = level_span<true>(gg.level, gg.preferred, -1, first);
  if (int(l) > first || int(l) < base || l >= tp.L || blockIdx.x * 32u >= tp.n_dom[l]) return;
  for (uint32_t c = threadIdx.x; c < gg.n_cliques; c += blockDim.x) {
    const grove_clique_t q = tb.cliques[gg.clique_off + c];
    sh.clq[c] = make_uint4(q.req_cpu_milli, q.req_mem_mib, q.req_gpu,
                           uint32_t(q.min_replicas) | (uint32_t(q.replicas) << 8) | (uint32_t(q.level) << 16) |
                               (GROVE_CLIQUE_PREFERRED(q.scope) << 24));
    sh.sig[c] = tb.cinfo[gg.clique_off + c].sig;
  }
  for (uint32_t si = threadIdx.x; si < gg.n_scopes; si += blockDim.x) sh.scopes[si] = tb.scopes[gg.scope_off + si];
  if (threadIdx.x == 0) s_bits = 0;
  __syncthreads();
  const uint32_t j = threadIdx.x >> 2, d = blockIdx.x * 32 + j;   // lanes 4j .. 4j + 3 of a warp share domain d
  bool plaus = d < tp.n_dom[l];
  if (plaus) {
    const uint32_t lo = __ldg(tp.dom_lo[l] + d), hi = __ldg(tp.dom_hi[l] + d);
    for (uint32_t si = slot; si < gg.n_scopes && plaus; si += 4) plaus = scope_ok(tp, rx, sh, sh.scopes[si], lo, hi, int(l), d);
  }
  plaus = plaus & bool(__shfl_xor_sync(kFull, uint32_t(plaus), 1));
  plaus = plaus & bool(__shfl_xor_sync(kFull, uint32_t(plaus), 2));
  const uint32_t b = __ballot_sync(kFull, plaus && slot == 0);
  if (lane == 0) {
    uint32_t bits = 0;
#pragma unroll
    for (uint32_t k = 0; k < 8; ++k) bits |= ((b >> (4 * k)) & 1u) << k;
    atomicOr(&s_bits, bits << (warp * 8));
  }
  __syncthreads();
  if (threadIdx.x == 0) const_cast<uint32_t*>(rx.shape_bits)[size_t(shape) * rx.pl_words + ((rx.pl_off[l] + blockIdx.x * 32) >> 5)] = s_bits;
}

// entry i of the round's evaluations: the heavy gangs of the list (from its head), the light ones (from its tail), then the new
// entrants of the window (ranks [kEntryLo, kHi): never evaluated, they need no list entry).  relax.cuh k_detect builds the list.
__device__ __forceinline__ uint32_t eval_list_at(const Relax& rx, const Tables& tb, uint32_t i) {
  const uint32_t nh = rx.ctl[kNHeavy], nl = rx.ctl[kNLight];
  if (i < nh) return rx.eval_list[i];
  if (i - nh < nl) return rx.eval_list[tb.G - 1u - (i - nh)];
  return tb.by_rank[rx.ctl[kEntryLo] + (i - nh - nl)];
}

// K3 evaluators: kW warps share ONE gang.  The candidates of the gang's level are pre-filtered 1024 at a time by all
// warps (a lane each); the plausible ones are then attempted kW at a time, a warp each, and the lowest successful
// candidate IN ORDER is the answer -- exactly what trying them one after the other gives, minus the waiting.  kW = 1
// while a round has many gangs (what matters is gangs in flight), 8 when it has few (what matters is the
// latency of the slowest gang: a round lasts as long as its slowest evaluation).
// Two roles in one launch per round (k_eval below): the LIGHT gangs (the tail of the list: most gangs, answered by their
// first or second candidate) a warp each -- every resident warp does useful work --, the HEAVY ones (the head: gangs whose
// last evaluation needed many attempts) kW warps each.  A light evaluation that is still unanswered after `max_att` attempts
// gives up (kEvalDeferred): the gang stays dirty and comes back as a heavy one next round, instead of holding the round up.
// Writes the "nxt" scratch of the gang.
constexpr uint32_t kEvalDeferred = 0xFFu;   // nxt_tstate: no result this round
constexpr int kHeavyWarps = 8;
// the shared state of one evaluator
template <int kW>
struct EvalShared {
  GangShared shs[kW];
  int4 s_view[kW][kStageMax];
  uint32_t s_vflag[kW][kStageMax];
  alignas(16) uint8_t s_rk[kW][kStageMax + 256];
  uint32_t s_plaus[32];                 // plausible candidates of the current 1024-candidate chunk, in order
  uint32_t s_cl[kW][32], s_ch[kW][32];  // node ranges of the first chunk's candidates (kW runs of 32)
  uint32_t s_win, s_ext, s_att, s_npl;
};
constexpr uint32_t kEvalThreads = kHeavyWarps * 32;
constexpr size_t kEvalSmem = sizeof(EvalShared<kHeavyWarps>) > kHeavyWarps * sizeof(EvalShared<1>) ? sizeof(EvalShared<kHeavyWarps>)
                                                                                                    : kHeavyWarps * sizeof(EvalShared<1>);

// the barrier of one evaluator: the CTA for the heavy role, the warp for the light one (its warps finish different numbers of gangs)
template <int kW>
__device__ __forceinline__ void group_sync() {
  if constexpr (kW == 1) __syncwarp(); else __syncthreads();
}

template <bool kPref, int kW, bool kHeavy>
__device__ __forceinline__ void eval_role(const Topo& tp, const Tables& tb, const Relax& rx, uint32_t max_att, EvalShared<kW>& es,
                                          uint32_t slot, uint32_t n_slots) {
  const uint32_t lane = threadIdx.x & 31, warp = kW == 1 ? 0u : threadIdx.x >> 5, tid = warp * 32 + lane;
  const uint32_t n_eval = rx.ctl[kNEval], n_heavy = rx.ctl[kNHeavy];
  GangShared& sh = es.shs[warp];
  const uint32_t seg_lo = kHeavy ? 0u : n_heavy, seg_hi = kHeavy ? n_heavy : n_eval;
  for (uint32_t ei = seg_lo + slot; ei < seg_hi; ei += n_slots) {
    const uint32_t gi = eval_list_at(rx, tb, ei);
    const grove_gang_t gg = tb.gangs[gi];
    const GangInfo info = tb.ginfo[gi];
    group_sync<kW>();   // the previous gang's shared state is no longer read
    // the gang's cliques and scopes (a lane each), the words of the re-evaluation shortcut and the base gang's rank are asked for
    // BEFORE anything looks at them: one L2 round trip for all of them instead of one per question
    const bool has_c = lane < gg.n_cliques, has_s = lane < gg.n_scopes;
    const grove_clique_t q0 = has_c ? tb.cliques[gg.clique_off + lane] : grove_clique_t{};
    const CliqueInfo ci0 = has_c ? tb.cinfo[gg.clique_off + lane] : CliqueInfo{};
    const grove_scope_t sc0 = has_s ? tb.scopes[gg.scope_off + lane] : grove_scope_t{};
    const uint32_t round_now = rx.ctl[kRound];
    const uint32_t le = rx.last_eval[gi], fu_word = rx.fail_upto[gi], ext_word = rx.extent[gi];
    // ---- gangs that need no packing
    uint32_t trivial = 0;
    if (gg.flags & GROVE_GANG_GATED) trivial = GROVE_GANG_GATED_SKIP;
    else if (gg.base_gang != GROVE_NONE_U32) {
      // considered at its own turn: the base gang must have been admitted before it (final, or tentatively so far)
      const uint32_t brank = tb.ginfo[gg.base_gang].order;
      uint32_t bs = GROVE_GANG_REJECTED;
      if (brank < info.order) bs = rx.tstate[gg.base_gang];   // final for ranks below the front; 0 (not evaluated yet) counts as not admitted: its first result marks us dirty
      if (bs != GROVE_GANG_ADMITTED) trivial = GROVE_GANG_BASE_REJECTED;
    }
    if (trivial) {
      if (tid == 0) {
        rx.nxt_tstate[gi] = uint8_t(trivial); rx.nxt_n[gi] = 0; rx.nxt_info[gi] = 0xFFu; rx.nxt_glo[gi] = GROVE_NONE_U32; rx.nxt_extent[gi] = 0;
      }
      for (uint32_t si = tid; si < gg.n_scopes; si += kW * 32) { rx.nxt_sc_lvl[gg.scope_off + si] = 0xFFu; rx.nxt_sc_lo[gg.scope_off + si] = GROVE_NONE_U32; }
      continue;
    }
    GangRegs g;
    g.a = info.anchor; g.L = tp.L; g.n = tp.n; g.rank = info.order;
#pragma unroll
    for (int l = 0; l < GROVE_MAX_LEVELS; ++l) { g.anc_lo[l] = info.anc_lo[l]; g.anc_hi[l] = info.anc_hi[l]; }
    if (has_c) {   // every warp keeps its own copy: attempts run independently (GROVE_MAX_GANG_CLIQUES = 32: a lane each)
      const uint32_t c = lane;
      const grove_clique_t q = q0;
      const CliqueInfo ci = ci0;
      sh.clq[c] = make_uint4(q.req_cpu_milli, q.req_mem_mib, q.req_gpu,
                             uint32_t(q.min_replicas) | (uint32_t(q.replicas) << 8) | (uint32_t(q.level) << 16) |
                                 (GROVE_CLIQUE_PREFERRED(q.scope) << 24));
      sh.rcp[c] = make_float4(q.req_cpu_milli ? 1.0f / float(q.req_cpu_milli) : 0.f, q.req_mem_mib ? 1.0f / float(q.req_mem_mib) : 0.f,
                              q.req_gpu ? 1.0f / float(q.req_gpu) : 0.f, 0.f);
      sh.sig[c] = ci.sig; sh.smask[c] = uint32_t(q.class_mask) | (ci.need_depth << 16);
      sh.Hlo[c] = 0; sh.Hhi[c] = 0; sh.c_got[c] = -1;
    }
    if (has_s) { sh.scopes[lane] = sc0; sh.s_got[lane] = -1; sh.s_lo[lane] = 0; }
    if (tid == 0) { es.s_win = GROVE_NONE_U32; es.s_ext = 0; es.s_att = 0; es.s_npl = 0; }
    group_sync<kW>();
    // A candidate that failed in the gang's last evaluation fails again unless a claim was withdrawn inside it since: views only
    // shrink otherwise (claims are added, settled claims move into the committed state).  So a re-evaluation skips the
    // candidates in front of its last answer that no withdrawal touched -- gangs that meet a nearly full cluster would
    // otherwise re-run dozens of failing attempts every round.  (Single candidate level only.)
    Ev<kPref> ev(tp, rx, sh, g, lane);                         // candidates of any size, node state from L2
    EvS<kPref> evs(tp, rx, sh, g, lane, es.s_view[warp], es.s_vflag[warp], es.s_rk[warp]);         // candidates of <= kStageMax nodes, node state staged in shared memory
    bool staged = false;  // the winning attempt ran on evs
    bool won = false;     // this warp holds the answer
    bool done = false;    // uniform over the evaluator
    int g_got = -1; uint32_t g_lo = 0;
    const long long t0 = rx.dbg ? clock64() : 0;
    // candidate levels: the Preferred level first (if any), widened level by level up to the Required one
    // (gl == -1: the whole cluster as a single candidate)
    int gfirst;
    const int gbase = level_span<kPref>(gg.level, gg.preferred, -1, gfirst);
    int gl = gfirst;
    const uint32_t fu = (le && gfirst == gbase && gfirst >= 0) ? fu_word : 0u;
    uint32_t k_won = 0;
    bool gave_up = false;
    do {
      if (gl < 0) {
        staged = false;
        if (warp == 0) {
          won = place_in(ev, gg.n_scopes, 0, tp.n, -1);
          if (won) { g_got = -1; g_lo = 0; if (lane == 0) es.s_win = 0; }
          if (lane == 0) es.s_att += 1;
        }
        group_sync<kW>();
        done = es.s_win != GROVE_NONE_U32;
      } else {
        // candidate domains of level gl in score order: up to kMaxPieces ranges of domain indices
        uint32_t r0[kMaxPieces], rcnt[kMaxPieces], D = 0;
        {
          uint32_t plo[kMaxPieces], phi[kMaxPieces];
          const int npc = make_pieces(g, 0, tp.n, uint32_t(gl), plo, phi);
          for (int p = 0; p < kMaxPieces; ++p) {
            r0[p] = 0; rcnt[p] = 0;
            if (p < npc) { r0[p] = __ldg(tp.next_dom[gl] + plo[p]); rcnt[p] = __ldg(tp.next_dom[gl] + phi[p]) - r0[p]; D += rcnt[p]; }
          }
        }
        auto cand = [&](uint32_t k, uint32_t& dl, uint32_t& dh) -> uint32_t {   // k-th candidate in order -> its domain
          uint32_t d = 0, rem = k;
#pragma unroll
          for (int p = 0; p < kMaxPieces; ++p) { if (rem < rcnt[p]) { d = r0[p] + rem; break; } rem -= rcnt[p]; }
          dl = __ldg(tp.dom_lo[gl] + d); dh = __ldg(tp.dom_hi[gl] + d);
          return d;
        };
        // candidates are taken in chunks that grow (kW x 32, then up to 1024): most gangs succeed among the first few
        for (uint32_t base = 0, nchunk = kW; base < D && !done && !gave_up; base += nchunk * 32, nchunk = min(32u, nchunk * 4u)) {
          // pre-filter: nchunk runs of 32 candidates, dealt to the warps
          for (uint32_t c = warp; c < nchunk; c += kW) {
            const uint32_t k = base + c * 32 + lane;
            bool plaus = false;
            if (k < D) {
              // the candidate's node range is fetched together with its pre-filter bit (the attempt would otherwise pay one more
              // L2 round trip for it); the first chunk's ranges wait in shared memory
              uint32_t dl, dh; const uint32_t d = cand(k, dl, dh);
              if (rx.shape_bits) {   // one bit per (shape, domain), refreshed with the capacity tables
                const uint32_t bit = rx.pl_off[gl] + d;
                plaus = (__ldg(rx.shape_bits + size_t(info.pad) * rx.pl_words + (bit >> 5)) >> (bit & 31u)) & 1u;
              } else {
                plaus = gang_plausible(tp, rx, sh, gg.n_scopes, dl, dh, gl, d);
              }
              if (base == 0) { es.s_cl[c][lane] = dl; es.s_ch[c][lane] = dh; }
              if (plaus && k < fu) {   // failed last time: worth another attempt only if somebody withdrew a claim in there since
                bool again = false;
                for (uint32_t w = dl >> 5; w <= (dh - 1u) >> 5; ++w) again |= __ldg(rx.rem_round + w) >= le;
                plaus = again;
              }
            }
            const uint32_t b = __ballot_sync(kFull, plaus);
            if (lane == 0) es.s_plaus[c] = b;
          }
          group_sync<kW>();
          uint32_t total = 0;
          for (uint32_t c = 0; c < nchunk; ++c) total += __popc(es.s_plaus[c]);
          if (tid == 0) es.s_npl += total;
          // attempts: kW plausible candidates at a time, in order, a warp each
          // while a round has many gangs the very first candidate is attempted by one warp alone: it usually succeeds,
          // and the other warps' attempts would be thrown away
          for (uint32_t j0 = 0; j0 < total && !done; j0 += uint32_t(kW)) {
            if (!kHeavy && max_att && es.s_att >= max_att) { gave_up = true; break; }   // uniform over the evaluator (read after its barrier)
            const uint32_t j = j0 + warp;
            bool ok = false; uint32_t dl = 0, dh = 0;
            if (j < total) {
              uint32_t rem = j, c = 0;   // the j-th set bit of the bitmap
              for (; c + 1 < nchunk; ++c) { const uint32_t pc = __popc(es.s_plaus[c]); if (rem < pc) break; rem -= pc; }
              uint32_t w = es.s_plaus[c];
              for (uint32_t i = 0; i < rem; ++i) w &= w - 1;
              const uint32_t kl = __ffs(w) - 1, k = base + c * 32 + kl;
              if (base == 0) { dl = es.s_cl[c][kl]; dh = es.s_ch[c][kl]; } else cand(k, dl, dh);
              staged = dh - dl <= kStageMax;
              ok = staged ? place_in(evs, gg.n_scopes, dl, dh, gl) : place_in(ev, gg.n_scopes, dl, dh, gl);
              if (lane == 0) { atomicAdd(&es.s_att, 1u); if (ok) atomicMin(&es.s_win, j); }
              if (ok) k_won = k;
            }
            group_sync<kW>();
            const uint32_t win = es.s_win;
            if (win != GROVE_NONE_U32) { done = true; won = ok && win == j; if (won) { g_got = gl; g_lo = dl; } }
          }
          group_sync<kW>();   // es.s_plaus is rewritten by the next chunk
        }
      }
    } while (kPref && !done && !gave_up && --gl >= gbase);
    // what any of the attempts may have read (attempts past the winner only widen it)
    if (lane == 0) atomicMax(&es.s_ext, max(max(ev.ext, evs.ext), fu ? ext_word : 0u));   // skipped candidates were read by the last evaluation
    group_sync<kW>();
    if (tid == 0) rx.last_att[gi] = uint8_t(gave_up ? 255u : min(254u, es.s_att));
    if (gave_up) {   // no result this round: k_apply keeps the gang dirty
      if (tid == 0) rx.nxt_tstate[gi] = uint8_t(kEvalDeferred);
      continue;
    }
    if (rx.dbg && tid == 0) {
      const uint32_t cyc = uint32_t(clock64() - t0);
      rx.dbg[gi * 8 + 0] += 1; rx.dbg[gi * 8 + 1] += es.s_npl; rx.dbg[gi * 8 + 2] += es.s_att;
      rx.dbg[gi * 8 + 3] = max(rx.dbg[gi * 8 + 3], cyc); rx.dbg[gi * 8 + 4] = cyc; rx.dbg[gi * 8 + 5] = es.s_att; rx.dbg[gi * 8 + 6] = es.s_npl; rx.dbg[gi * 8 + 7] = rx.ctl[kRound];
      // warp 0's own phases, summed over the cycle: staging, sub-domain pre-filter, packing, attempts staged
      atomicAdd(rx.dbg + tb.G * 8 + 0, evs.t_stage); atomicAdd(rx.dbg + tb.G * 8 + 1, evs.t_pre); atomicAdd(rx.dbg + tb.G * 8 + 2, evs.t_pack);
      atomicAdd(rx.dbg + tb.G * 8 + 3, evs.n_stage); atomicAdd(rx.dbg + tb.G * 8 + 4, cyc); atomicAdd(rx.dbg + tb.G * 8 + 5, 1u);
      atomicAdd(rx.dbg + tb.G * 8 + 6, evs.t_st2); atomicAdd(rx.dbg + tb.G * 8 + 7, evs.t_st3);
    }
    if (!done) {
      if (tid == 0) {
        rx.last_eval[gi] = round_now; rx.fail_upto[gi] = kFull;   // every candidate failed
        rx.nxt_tstate[gi] = GROVE_GANG_REJECTED; rx.nxt_n[gi] = 0; rx.nxt_info[gi] = 0xFFu; rx.nxt_glo[gi] = GROVE_NONE_U32;
        rx.nxt_extent[gi] = es.s_ext;
      }
      for (uint32_t si = tid; si < gg.n_scopes; si += kW * 32) { rx.nxt_sc_lvl[gg.scope_off + si] = 0xFFu; rx.nxt_sc_lo[gg.scope_off + si] = GROVE_NONE_U32; }
      continue;
    }
    if (!won) continue;   // warp-uniform: the winner finishes alone
    // surplus beyond MinReplicas (best effort, podgang.go:80-83), inside the domain each clique was packed into
    for (uint32_t cr = 0; cr < gg.n_cliques; ++cr) {
      const uint32_t w = sh.clq[cr].w;
      const uint32_t mn = w & 0xFFu, rp = (w >> 8) & 0xFFu;
      if (rp > mn) { if (staged) evs.take(cr, sh.Hlo[cr], sh.Hhi[cr], rp - mn); else ev.take(cr, sh.Hlo[cr], sh.Hhi[cr], rp - mn); }
    }
    __syncwarp();
    const uint32_t n_ent = staged ? evs.np : ev.np;
    // PlacementScore: levels honoured / levels asked for, over the gang, its scopes and its cliques
    uint32_t num = 0, den = 0;
    if (lane == 0) score_unit(gg.level, gg.preferred, g_got, num, den);
    if (lane < gg.n_scopes) {
      const grove_scope_t s = sh.scopes[lane];
      score_unit(s.level, s.preferred1 ? uint32_t(s.preferred1) - 1u : uint32_t(GROVE_LEVEL_NONE), int(sh.s_got[lane]), num, den);
    }
    if (lane < gg.n_cliques) {
      const uint32_t w = sh.clq[lane].w;
      score_unit((w >> 16) & 0xFFu, w >> 24, int(sh.c_got[lane]), num, den);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { num += __shfl_xor_sync(kFull, num, o); den += __shfl_xor_sync(kFull, den, o); }
    if (den == 0) { num = 1; den = 1; }
    for (uint32_t i = lane; i < n_ent; i += 32) {
      rx.nxt_node[info.pod_off + i] = sh.ent_node[i];
      rx.nxt_meta[info.pod_off + i] = sh.ent_meta[i];
    }
    for (uint32_t si = lane; si < gg.n_scopes; si += 32) {
      const bool own = int(sh.s_got[si]) > g_got;   // a scope packed at the gang's own level has no domain of its own
      rx.nxt_sc_lvl[gg.scope_off + si] = own ? uint8_t(sh.s_got[si]) : uint8_t(0xFFu);
      rx.nxt_sc_lo[gg.scope_off + si] = own ? sh.s_lo[si] : GROVE_NONE_U32;
    }
    if (lane == 0) {
      rx.last_eval[gi] = round_now; rx.fail_upto[gi] = g_got >= 0 ? k_won : 0u;
      rx.nxt_tstate[gi] = GROVE_GANG_ADMITTED; rx.nxt_n[gi] = uint16_t(n_ent);
      rx.nxt_info[gi] = (g_got >= 0 ? uint32_t(g_got) : 0xFFu) | (num << 8) | (den << 20);
      rx.nxt_glo[gi] = g_got >= 0 ? g_lo : GROVE_NONE_U32;
      rx.nxt_extent[gi] = max(max(ev.ext, evs.ext), es.s_ext);   // the surplus pass above may have read further
    }
  }
}

// One launch per round, 256-thread CTAs.  CTAs [0, heavy_ctas) take the heavy role: kHeavyWarps warps share a gang, the list is
// read from its head.  The others take the light role: every warp is an evaluator of its own (grid-strided over the warps of the
// light CTAs) with the max_att give-up.  Heavy CTAs have the low indices so that they are dispatched first.  The role is
// uniform over the CTA; each role's shared state is carved out of one dynamic buffer of kEvalSmem bytes.
template <bool kPref>
__global__ void __launch_bounds__(kEvalThreads, 2) k_eval(Topo tp, Tables tb, Relax rx, uint32_t heavy_ctas, uint32_t max_att) {
  extern __shared__ __align__(16) unsigned char eval_smem[];
  pdl_begin();
  if (rx.ctl[kDone]) return;
  if (blockIdx.x < heavy_ctas) {
    eval_role<kPref, kHeavyWarps, true>(tp, tb, rx, 0u, *reinterpret_cast<EvalShared<kHeavyWarps>*>(eval_smem), blockIdx.x, heavy_ctas);
  } else {
    const uint32_t warp = threadIdx.x >> 5;
    eval_role<kPref, 1, false>(tp, tb, rx, max_att, reinterpret_cast<EvalShared<1>*>(eval_smem)[warp],
                               (blockIdx.x - heavy_ctas) * kHeavyWarps + warp, (gridDim.x - heavy_ctas) * kHeavyWarps);
  }
}

}  // namespace grove
