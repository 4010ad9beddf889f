// relax.cuh -- the relaxation that turns per-gang evaluations into the sequential cycle, and the output kernels.
#pragma once
#include "common.cuh"
#include "admit.cuh"

namespace grove {
// ------------------------------------------------------------------------------------------------
// The cycle's result is defined sequentially: gang of rank 0, then rank 1, ... each against the state the
// earlier ones left.  Equivalently: the unique assignment in which EVERY gang's placement equals its
// evaluation against (committed state - claims of all gangs that rank before it).  The engine iterates
// towards that fixed point with all gangs of a window at once:
//
//   round:  k_eval     (admit.cuh) the gangs of the window [front, hi) that were never evaluated (the new entrants) or whose
//                      view changed (the list k_detect left), each against its view -> "nxt" scratch   [reads claims]
//           k_apply    a changed result withdraws the gang's old claims and publishes the new
//                      ones; every withdrawal / addition leaves a stamp (round tag | rank)   [writes claims]
//           k_detect   whose view changed?  a gang is dirty if a LOWER rank added a claim on a node it uses
//                      (capacity it counted on is gone), withdrew a claim in front of its extent (capacity it did
//                      not see is back), or its base gang's result changed.  front' = lowest dirty rank.
//                      Gangs of rank < front' are final: every rank before them is final and their last evaluation saw
//                      exactly those claims.  The last CTA of k_detect advances the window.
//   now and then (before a capacity-table rebuild, and when the cycle ends):
//           k_fold     the claims of the final gangs are folded into the committed state (until then they simply stay
//                      claims: every gang of the window ranks after them and subtracts them anyway).
//
// Why it is exact: by induction on rank, a gang that is not dirty while everything before it is final holds the
// sequential answer.  Why it terminates: the lowest gang of the window is never dirty after its evaluation.
// Monotonicity does the rest of the work: resources only shrink inside a cycle, so additions by lower ranks
// can only matter on the nodes a gang actually uses, and infeasible candidates stay infeasible.
// Nothing here decides a result by arrival order: claims are sums, stamps are minima.
// ------------------------------------------------------------------------------------------------

// The state a cycle starts from, in ONE launch (it used to be two dozen memsets and a blocking upload of the control words: a tenth
// of a millisecond of launch latencies in front of every cycle)
// (n_cap: words of the capacity sum / max tables, which the first k_fit accumulates into)
__global__ void __launch_bounds__(256) k_reset(Relax rx, uint32_t G, uint32_t NS, uint32_t npad, uint32_t words, uint32_t hi0, uint32_t n_cap) {
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  for (uint32_t i = tid; i < n_cap; i += nt) { rx.capsum[i] = 0; rx.capmax[i] = 0; }
  const uint4 ones = make_uint4(kFull, kFull, kFull, kFull);
  for (size_t i = tid; i < size_t(npad) * kClaimSlots; i += nt) rx.claims[i] = ones;
  for (uint32_t i = tid; i < npad; i += nt) { rx.ctot[i] = make_int4(0, 0, 0, 0); rx.cmaxr[i] = 0; rx.ovf_head[i] = 0; rx.add_stamp[i] = kFull; }
  for (uint32_t i = tid; i < npad / 4; i += nt) rx.nlive[i] = 0;
  for (uint32_t i = tid; i < words; i += nt) { rx.rem_stamp[i] = kFull; rx.rem_round[i] = 0; }
  for (uint32_t i = tid; i < G; i += nt) {
    rx.state[i] = 0; rx.tstate[i] = 0; rx.dirty[i] = 0; rx.last_att[i] = 0; rx.cur_n[i] = 0;
    rx.chg_round[i] = 0; rx.cur_info[i] = 0; rx.cur_glo[i] = 0; rx.extent[i] = 0; rx.last_eval[i] = 0;
  }
  for (uint32_t i = tid; i < NS; i += nt) { rx.sc_lvl[i] = 0xFFu; rx.sc_lo[i] = kFull; }
  if (tid < kCtlWords) {
    uint32_t v = 0;
    if (tid == kHi || tid == kMinDirty || tid == kNEval) v = hi0;   // the first round evaluates the first window's worth of new entrants
    if (tid == kRound) v = 1;
    if (tid == kRemAny) v = kFull;
    if (tid == kDone) v = G == 0;
    rx.ctl[tid] = v;
  }
}

// ---- claims --------------------------------------------------------------------------------------------
__device__ __forceinline__ void nlive_add(uint32_t* nlive, uint32_t n, int delta) {
  const uint32_t sh = (n & 3u) * 8u;
  if (delta > 0) atomicAdd(nlive + (n >> 2), 1u << sh); else atomicSub(nlive + (n >> 2), 1u << sh);
}

// the per-node total of all live claims follows every claim that comes or goes (gpw = gpu | pods << 16, sign = +1 / -1)
__device__ __forceinline__ void ctot_add(const Relax& rx, uint32_t n, int cpu, int mem, uint32_t gpw, int sign) {
  int* t = reinterpret_cast<int*>(rx.ctot + n);
  if (cpu) atomicAdd(t + 0, cpu);
  if (mem) atomicAdd(t + 1, mem);
  if (gpw & 0xFFFFu) atomicAdd(t + 2, sign * int(gpw & 0xFFFFu));
  atomicAdd(t + 3, sign * int(gpw >> 16));
}

// withdraw ONE claim slot of `rank` on node n (the caller owns exactly one per entry run)
__device__ __forceinline__ void claim_remove(const Relax& rx, uint32_t n, uint32_t rank) {
  uint32_t* line = reinterpret_cast<uint32_t*>(rx.claims + size_t(n) * kClaimSlots);
  // look first (one cache line), then take: an atomic per slot would be a chain of L2 round trips
  uint32_t own = 0;
#pragma unroll
  for (uint32_t s = 0; s < kClaimSlots; ++s) own |= uint32_t(__ldcg(line + 4 * s) == rank) << s;
  for (; own; own &= own - 1) {
    const uint32_t s = __ffs(own) - 1;
    // the amounts are read while the slot is still ours: once it is free another gang may take and rewrite it
    const uint32_t cpu = __ldcg(line + 4 * s + 1), mem = __ldcg(line + 4 * s + 2), gpw = __ldcg(line + 4 * s + 3);
    if (atomicCAS(line + 4 * s, rank, kClaimEmpty) == rank) {   // (another lane of this gang may have taken it)
      ctot_add(rx, n, -int(cpu), -int(mem), gpw, -1);
      nlive_add(rx.nlive, n, -1);
      return;
    }
  }
  for (uint32_t i = *reinterpret_cast<volatile uint32_t*>(rx.ovf_head + n); i; i = rx.ovf_next[i - 1]) {
    uint32_t* e = reinterpret_cast<uint32_t*>(rx.ovf_claim + i - 1);
    if (__ldcg(e) != rank) continue;
    const uint32_t cpu = __ldcg(e + 1), mem = __ldcg(e + 2), gpw = __ldcg(e + 3);
    if (atomicCAS(e, rank, kClaimEmpty) == rank) { ctot_add(rx, n, -int(cpu), -int(mem), gpw, -1); return; }
  }
}

__device__ __forceinline__ void claim_add(const Relax& rx, uint32_t n, uint32_t rank, uint32_t cpu, uint32_t mem, uint32_t gpw) {
  uint32_t* line = reinterpret_cast<uint32_t*>(rx.claims + size_t(n) * kClaimSlots);
  ctot_add(rx, n, int(cpu), int(mem), gpw, +1);
  atomicMax(rx.cmaxr + n, rank);
  for (int pass = 0; pass < 3; ++pass) {   // look first, then take; somebody else may win the slot: look again
    uint32_t freeb = 0;
#pragma unroll
    for (uint32_t s = 0; s < kClaimSlots; ++s) freeb |= uint32_t(__ldcg(line + 4 * s) == kClaimEmpty) << s;
    if (!freeb) break;
    for (; freeb; freeb &= freeb - 1) {
      const uint32_t s = __ffs(freeb) - 1;
      if (atomicCAS(line + 4 * s, kClaimEmpty, rank) == kClaimEmpty) {
        line[4 * s + 1] = cpu; line[4 * s + 2] = mem; line[4 * s + 3] = gpw;
        nlive_add(rx.nlive, n, +1);
        return;
      }
    }
  }
  // more than kClaimSlots gangs lean on this node: its overflow chain.  A dead entry of the chain is revived first;
  // otherwise a pool entry is pushed on the chain's head (entries never leave a chain during a cycle)
  for (uint32_t i = *reinterpret_cast<volatile uint32_t*>(rx.ovf_head + n); i; i = rx.ovf_next[i - 1]) {
    uint32_t* e = reinterpret_cast<uint32_t*>(rx.ovf_claim + i - 1);
    if (atomicCAS(e, kClaimEmpty, rank) == kClaimEmpty) { e[1] = cpu; e[2] = mem; e[3] = gpw; return; }
  }
  const uint32_t i = atomicAdd(rx.ctl + kOvfCount, 1u);
  if (i >= rx.ovf_cap) return;   // pool exhausted: the host sees the count and fails the cycle
  rx.ovf_claim[i] = make_uint4(rank, cpu, mem, gpw);
  uint32_t old = *reinterpret_cast<volatile uint32_t*>(rx.ovf_head + n);
  for (;;) {
    rx.ovf_next[i] = old;
    __threadfence();
    const uint32_t seen = atomicCAS(rx.ovf_head + n, old, i + 1u);
    if (seen == old) break;
    old = seen;
  }
  atomicOr(rx.nlive + (n >> 2), kHasOvf << ((n & 3u) * 8u));
}

// entry i of a placement starts a run of pods of one clique on one node; returns its length (0 = not a head)
__device__ __forceinline__ uint32_t run_length(const uint32_t* node, const uint16_t* meta, uint32_t i, uint32_t cnt) {
  if (i && node[i - 1] == node[i] && meta[i - 1] == meta[i]) return 0;
  uint32_t t = 1;
  while (i + t < cnt && node[i + t] == node[i] && meta[i + t] == meta[i]) ++t;
  return t;
}

// one warp per evaluated gang: publish a changed result
__global__ void __launch_bounds__(256) k_apply(Tables tb, Relax rx) {
  const uint32_t lane = threadIdx.x & 31;
  pdl_begin();
  if (rx.ctl[kDone]) return;
  const uint32_t n_eval = rx.ctl[kNEval], round = rx.ctl[kRound];
  const uint32_t nw = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t ei = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; ei < n_eval; ei += nw) {
    const uint32_t g = eval_list_at(rx, tb, ei);
    // every word the comparison needs is asked for at once (a chain of `||` would fetch them one L2 round trip after the other)
    const grove_gang_t gg = tb.gangs[g];
    const uint32_t po = tb.ginfo[g].pod_off, rank = tb.ginfo[g].order;
    const uint32_t ot = rx.tstate[g], nt = rx.nxt_tstate[g];
    const uint32_t c_n = rx.cur_n[g], n_n = rx.nxt_n[g], c_info = rx.cur_info[g], n_info = rx.nxt_info[g], c_glo = rx.cur_glo[g], n_glo = rx.nxt_glo[g];
    const uint32_t n_ext = rx.nxt_extent[g];
    if (lane == 0) rx.dirty[g] = nt == kEvalDeferred;   // the only dirtiness that outlives a round: no result yet
    if (nt == kEvalDeferred) {   // the light evaluation gave up: no result, the gang is evaluated again (as a heavy one) next round
      if (lane == 0) atomicMin(rx.ctl + kMinDirty, rank);
      continue;
    }
    const uint32_t on = ot == GROVE_GANG_ADMITTED ? c_n : 0u, nn = nt == GROVE_GANG_ADMITTED ? n_n : 0u;
    bool diff = (ot != nt) | (on != nn) | (c_info != n_info) | (c_glo != n_glo);
    if (!diff) {
      for (uint32_t i = lane; i < nn; i += 32) {
        const uint32_t a = rx.ent_node[po + i], b = rx.nxt_node[po + i]; const uint16_t c = rx.ent_meta[po + i], d = rx.nxt_meta[po + i];
        diff |= (a != b) | (c != d);
      }
      for (uint32_t si = lane; si < gg.n_scopes; si += 32) {
        const uint8_t a = rx.sc_lvl[gg.scope_off + si], b = rx.nxt_sc_lvl[gg.scope_off + si]; const uint32_t c = rx.sc_lo[gg.scope_off + si], d = rx.nxt_sc_lo[gg.scope_off + si];
        diff |= (a != b) | (c != d);
      }
    }
    diff = __any_sync(kFull, diff);
    if (lane == 0) rx.extent[g] = n_ext;   // what the LATEST evaluation read, changed result or not
    if (!diff) continue;
    const uint32_t stamp = make_stamp(round, rank);
    // withdraw the old claims
    for (uint32_t i = lane; i < on; i += 32) {
      if (!run_length(rx.ent_node + po, rx.ent_meta + po, i, on)) continue;
      const uint32_t n = rx.ent_node[po + i];
      claim_remove(rx, n, rank);
      atomicMin(rx.rem_stamp + (n >> 5), stamp);
      atomicMax(rx.rem_round + (n >> 5), round);
    }
    if (on && lane == 0) atomicMin(rx.ctl + kRemAny, stamp);
    __syncwarp();
    // publish the new ones
    for (uint32_t i = lane; i < nn; i += 32) {
      const uint32_t n = rx.nxt_node[po + i]; const uint16_t m = rx.nxt_meta[po + i];
      const uint32_t t = run_length(rx.nxt_node + po, rx.nxt_meta + po, i, nn);
      if (t) {
        const grove_clique_t q = tb.cliques[gg.clique_off + m];
        claim_add(rx, n, rank, t * q.req_cpu_milli, t * q.req_mem_mib, t * uint32_t(q.req_gpu) | (t << 16));
        atomicMin(rx.add_stamp + n, stamp);
      }
    }
    __syncwarp();
    for (uint32_t i = lane; i < nn; i += 32) { rx.ent_node[po + i] = rx.nxt_node[po + i]; rx.ent_meta[po + i] = rx.nxt_meta[po + i]; }
    for (uint32_t si = lane; si < gg.n_scopes; si += 32) { rx.sc_lvl[gg.scope_off + si] = rx.nxt_sc_lvl[gg.scope_off + si]; rx.sc_lo[gg.scope_off + si] = rx.nxt_sc_lo[gg.scope_off + si]; }
    if (lane == 0) {
      rx.tstate[g] = uint8_t(nt); rx.cur_n[g] = uint16_t(nn); rx.cur_info[g] = rx.nxt_info[g]; rx.cur_glo[g] = rx.nxt_glo[g];
      rx.chg_round[g] = round;
      atomicAdd(rx.ctl + kChanged, 1u);
    }
  }
}

// one warp per gang of the window: did its view change this round?
__global__ void __launch_bounds__(256) k_detect(Topo tp, Tables tb, Relax rx, uint32_t refresh_every) {
  __shared__ bool s_last;
  const uint32_t lane = threadIdx.x & 31;
  pdl_begin();
  if (rx.ctl[kDone]) return;   // uniform over the grid: set only by the last CTA of an earlier launch
  const uint32_t front = rx.ctl[kFront], hi = rx.ctl[kHi], round = rx.ctl[kRound];
  const uint32_t rem_any = rx.ctl[kRemAny];
  const uint32_t nw = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t p = front + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); p < hi; p += nw) {
    const uint32_t g = tb.by_rank[p];   // rank of g == p
    // the gang's words are asked for at once (conditions one after the other would fetch them one L2 round trip each)
    const uint32_t base = tb.gangs[g].base_gang;
    const uint32_t po = tb.ginfo[g].pod_off;
    const uint32_t ts = rx.tstate[g], cnt = rx.cur_n[g], ext = rx.extent[g];
    bool dirty = rx.dirty[g] != 0;   // its evaluation gave up this round (k_apply)
    const uint32_t first_node = (ts == GROVE_GANG_ADMITTED && lane < cnt) ? rx.ent_node[po + lane] : GROVE_NONE_U32;
    // its base gang's result changed
    if (base != GROVE_NONE_U32 && rx.chg_round[base] == round) dirty = true;
    // a lower rank newly claimed a node this gang uses
    if (ts == GROVE_GANG_ADMITTED) {
      if (first_node != GROVE_NONE_U32) dirty |= stamp_below(rx.add_stamp[first_node], round, p);
      for (uint32_t i = lane + 32; i < cnt; i += 32) dirty |= stamp_below(rx.add_stamp[rx.ent_node[po + i]], round, p);
    }
    dirty = __any_sync(kFull, dirty);
    // a lower rank withdrew a claim among the nodes the last evaluation may have read
    uint32_t left = ext;
    if (!dirty && left && stamp_below(rem_any, round, p)) {
      const GangInfo info = tb.ginfo[g];
      GangRegs gr;
      gr.a = info.anchor; gr.L = tp.L; gr.n = tp.n; gr.rank = p;
#pragma unroll
      for (int l = 0; l < GROVE_MAX_LEVELS; ++l) { gr.anc_lo[l] = info.anc_lo[l]; gr.anc_hi[l] = info.anc_hi[l]; }
      uint32_t plo[kMaxPieces], phi[kMaxPieces];
      const int npc = make_pieces(gr, 0, tp.n, tp.L, plo, phi);
      for (int k = 0; k < npc && left && !dirty; ++k) {
        const uint32_t len = min(phi[k] - plo[k], left);
        left -= len;
        const uint32_t g0 = plo[k] >> 5, g1 = (plo[k] + len - 1u) >> 5;
        bool hit = false;
        for (uint32_t w = g0 + lane; w <= g1; w += 32) hit |= stamp_below(rx.rem_stamp[w], round, p);
        dirty = __any_sync(kFull, hit);
      }
    }
    if (dirty && lane == 0) {
      atomicMin(rx.ctl + kMinDirty, p);
      // the next round's list.  Longest first: a round lasts as long as its slowest evaluation, so the gangs whose last evaluation
      // needed several attempts get kHeavyWarps warps (head of the list), the others a warp each (tail)
      if (rx.last_att[g] >= rx.heavy_att) rx.eval_list[atomicAdd(rx.ctl + kNHeavyNext, 1u)] = g;
      else rx.eval_list[tb.G - 1u - atomicAdd(rx.ctl + kNLightNext, 1u)] = g;
    }
  }
  // the last CTA to finish advances the window and resets the per-round control words
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(rx.ctl + kCtaDone, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    const uint32_t G = tb.G;
    const uint32_t nf = *reinterpret_cast<volatile uint32_t*>(rx.ctl + kMinDirty);
    // the window: at most `window` gangs beyond the settled prefix, at most `entry` new ones per round (gangs that meet
    // the claims of the ranks before them on their first evaluation pile up less on the same nodes)
    const uint32_t h2 = min(G, min(nf + rx.window, max(rx.ctl[kHi], nf) + rx.entry));
    const uint32_t old_hi = max(rx.ctl[kHi], nf);   // (nf <= hi always: the lowest dirty rank lies inside the window or is its end)
    const uint32_t nh = rx.ctl[kNHeavyNext], nl = rx.ctl[kNLightNext];
    rx.ctl[kEvals] += rx.ctl[kNEval];
    rx.ctl[kFront] = nf; rx.ctl[kHi] = h2; rx.ctl[kMinDirty] = h2; rx.ctl[kChanged] = 0;
    rx.ctl[kEntryLo] = old_hi; rx.ctl[kNHeavy] = nh; rx.ctl[kNLight] = nl; rx.ctl[kNEval] = nh + nl + (h2 - min(old_hi, h2));
    rx.ctl[kNHeavyNext] = 0; rx.ctl[kNLightNext] = 0;
    rx.ctl[kRound] += 1; rx.ctl[kRemAny] = kFull; rx.ctl[kCtaDone] = 0;
    rx.ctl[kDone] = nf >= G ? 1u : 0u;
    if (nf < G && nf - rx.ctl[kTablesAt] >= refresh_every) rx.ctl[kRefresh] = 1;
    __threadfence();
    if (rx.live) {
      volatile uint32_t* lv = rx.live;
      lv[kLiveFront] = nf; lv[kLiveDone] = nf >= G ? 1u : 0u; lv[kLiveRefresh] = rx.ctl[kRefresh]; lv[kLiveOvf] = rx.ctl[kOvfCount]; lv[kLiveEvals] = rx.ctl[kEvals];
      __threadfence_system();
      lv[kLiveRound] = rx.ctl[kRound];
    }
  }
}

// one warp per gang that became final since the last fold: its claims move into the committed state.  Not every round: the
// claims of final gangs are as good as committed for everybody who ranks after them, so the fold runs before a capacity-table
// rebuild (the tables are built from the committed state) and when the cycle ends; its last CTA then moves the marker.
// Before a rebuild (n_cap != 0) it also zeroes the capacity sum / max tables that k_fit accumulates into.
__global__ void __launch_bounds__(256) k_fold(Tables tb, Relax rx, uint4* nres, uint32_t n_cap) {
  __shared__ bool s_last;
  const uint32_t lane = threadIdx.x & 31;
  pdl_begin();
  const uint32_t lo = rx.ctl[kFolded], hi = rx.ctl[kFront];
  const uint32_t nw = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_cap; i += gridDim.x * blockDim.x) { rx.capsum[i] = 0; rx.capmax[i] = 0; }
  for (uint32_t p = lo + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); p < hi; p += nw) {
    const uint32_t g = tb.by_rank[p];
    const uint32_t t = rx.tstate[g];
    if (lane == 0) rx.state[g] = uint8_t(t);
    if (t != GROVE_GANG_ADMITTED) continue;
    const uint32_t po = tb.ginfo[g].pod_off, cnt = rx.cur_n[g], coff = tb.gangs[g].clique_off;
    for (uint32_t i = lane; i < cnt; i += 32) {
      const uint32_t len = run_length(rx.ent_node + po, rx.ent_meta + po, i, cnt);
      if (!len) continue;
      const uint32_t n = rx.ent_node[po + i];
      const grove_clique_t q = tb.cliques[coff + rx.ent_meta[po + i]];
      claim_remove(rx, n, p);
      uint32_t* r = reinterpret_cast<uint32_t*>(nres + n);
      if (q.req_cpu_milli) atomicSub(r + 0, len * q.req_cpu_milli);
      if (q.req_mem_mib) atomicSub(r + 1, len * q.req_mem_mib);
      atomicSub(r + 2, len * uint32_t(q.req_gpu) | (len << 16));
      atomicOr(rx.nlive + (n >> 2), kStale << ((n & 3u) * 8u));   // the capacity tables no longer describe this node
    }
  }
  // the last CTA moves the marker, once every CTA has read it (the counter is k_detect's: idle between its launches)
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(rx.ctl + kCtaDone, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last && threadIdx.x == 0) { rx.ctl[kFolded] = hi; rx.ctl[kCtaDone] = 0; }
}

// after a capacity-table build: the tables describe every node again
__global__ void k_clear_stale(Relax rx, uint32_t n_words) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_begin();
  if (i < n_words) rx.nlive[i] &= ~0x80808080u;
  if (i == 0) { rx.ctl[kTablesAt] = rx.ctl[kFront]; rx.ctl[kRefresh] = 0; rx.ctl[kFoldAny] = 0; }
}

// ------------------------------------------------------------------------------------------------
// outputs: compact the admitted gangs' entries into caller order / caller node indices
// ------------------------------------------------------------------------------------------------
// pass 1: per-CTA pod totals; pass 2 (one CTA): exclusive scan of the totals; pass 3: statuses with global offsets
constexpr int kFinThreads = 1024;

__global__ void __launch_bounds__(kFinThreads) k_fin_count(Tables tb, Relax rx, uint32_t* cta_tot) {
  __shared__ uint32_t s_w[32];
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t g = blockIdx.x * kFinThreads + tid;
  pdl_begin();
  uint32_t cnt = 0, adm = 0, rej = 0;
  if (g < tb.G) {
    const uint8_t st = rx.state[g];
    if (st == GROVE_GANG_ADMITTED) { cnt = rx.cur_n[g]; adm = 1; }
    rej = st == GROVE_GANG_REJECTED || st == GROVE_GANG_BASE_REJECTED;
  }
  uint32_t v = cnt | 0;   // three sums through one reduction each
#pragma unroll
  for (int o = 16; o; o >>= 1) { v += __shfl_xor_sync(kFull, v, o); adm += __shfl_xor_sync(kFull, adm, o); rej += __shfl_xor_sync(kFull, rej, o); }
  if (lane == 0) { s_w[warp] = v; atomicAdd(cta_tot + gridDim.x + 1, adm); atomicAdd(cta_tot + gridDim.x + 2, rej); }
  __syncthreads();
  if (warp == 0) {
    uint32_t t = s_w[lane];
#pragma unroll
    for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(kFull, t, o);
    if (lane == 0) cta_tot[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(1024) k_fin_scan(uint32_t* cta_tot, uint32_t n_cta, uint32_t* totals) {
  // n_cta <= 16384 gangs-per-CTA blocks; a single CTA scans them in chunks of 1024
  __shared__ uint32_t s_w[32];
  __shared__ uint32_t s_run;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_begin();
  if (tid == 0) s_run = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n_cta; base += 1024) {
    const uint32_t i = base + tid;
    const uint32_t v = i < n_cta ? cta_tot[i] : 0u;
    const uint32_t incl = warp_incl_scan(v, lane);
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) { const uint32_t w = s_w[lane]; const uint32_t s = warp_incl_scan(w, lane); s_w[lane] = s - w; }
    __syncthreads();
    const uint32_t excl = s_run + s_w[warp] + incl - v;
    if (i < n_cta) cta_tot[i] = excl;
    __syncthreads();
    if (tid == 1023) s_run = excl + v;
    __syncthreads();
  }
  if (tid == 0) { totals[0] = s_run; totals[1] = cta_tot[n_cta + 1]; totals[2] = cta_tot[n_cta + 2]; }
}

__global__ void __launch_bounds__(kFinThreads) k_fin_status(Tables tb, Relax rx, const uint32_t* __restrict__ cta_off,
                                                          const uint32_t* __restrict__ perm, grove_gang_status_t* status) {
  __shared__ uint32_t s_w[32];
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t g = blockIdx.x * kFinThreads + tid;
  pdl_begin();
  uint32_t cnt = 0; uint8_t st = 0;
  if (g < tb.G) { st = rx.state[g]; if (st == GROVE_GANG_ADMITTED) cnt = rx.cur_n[g]; }
  const uint32_t incl = warp_incl_scan(cnt, lane);
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  if (warp == 0) { const uint32_t w = s_w[lane]; const uint32_t s = warp_incl_scan(w, lane); s_w[lane] = s - w; }
  __syncthreads();
  if (g < tb.G) {
    grove_gang_status_t o;
    o.state = st; o.level = GROVE_LEVEL_NONE; o.reserved0 = 0; o.score_num = 0; o.score_den = 0;
    o.n_pods = cnt; o.placement_off = cta_off[blockIdx.x] + s_w[warp] + incl - cnt;
    o.domain_node = GROVE_NONE_U32; o.reserved1[0] = o.reserved1[1] = o.reserved1[2] = 0;
    if (st == GROVE_GANG_ADMITTED) {
      const uint32_t info = rx.cur_info[g];
      o.level = uint8_t(info & 0xFFu); o.score_num = uint16_t((info >> 8) & 0xFFFu); o.score_den = uint16_t(info >> 20);
      if ((info & 0xFFu) != GROVE_LEVEL_NONE) o.domain_node = perm[rx.cur_glo[g]];
    }
    status[g] = o;
  }
}

// one warp per gang: its entries -> caller node indices, at the offset k_fin_status assigned; its scopes' domains
__global__ void k_emit(Tables tb, Relax rx, const uint32_t* __restrict__ perm, const grove_gang_status_t* __restrict__ status,
                       grove_placement_t* out, grove_scope_status_t* scopes_out) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  pdl_begin();
  if (g >= tb.G) return;
  const grove_gang_status_t st = status[g];
  const grove_gang_t gg = tb.gangs[g];
  const bool adm = st.state == GROVE_GANG_ADMITTED;
  for (uint32_t si = lane; si < gg.n_scopes; si += 32) {
    grove_scope_status_t s;
    s.level = GROVE_LEVEL_NONE; s.reserved[0] = s.reserved[1] = s.reserved[2] = 0; s.domain_node = GROVE_NONE_U32;
    if (adm && rx.sc_lvl[gg.scope_off + si] != 0xFFu) { s.level = rx.sc_lvl[gg.scope_off + si]; s.domain_node = perm[rx.sc_lo[gg.scope_off + si]]; }
    scopes_out[gg.scope_off + si] = s;
  }
  if (!adm) return;
  const uint32_t po = tb.ginfo[g].pod_off;
  for (uint32_t i = lane; i < st.n_pods; i += 32) {
    grove_placement_t p;
    p.clique = gg.clique_off + rx.ent_meta[po + i];
    p.node = perm[rx.ent_node[po + i]];
    out[st.placement_off + i] = p;
  }
}

}  // namespace grove
