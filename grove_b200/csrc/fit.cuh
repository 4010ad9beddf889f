// fit.cuh -- K1: node x clique resource-fit bitmap with the per-signature capacity bytes, and their per-domain sums.
#pragma once
#include "common.cuh"

namespace grove {
// ------------------------------------------------------------------------------------------------
// K1: node x clique resource-fit bitmap.
// CTA = 1024 nodes (lane = node, record in registers) x a tile of kFitTile clique rows whose
// requirements are staged in shared memory.  One __ballot_sync per (warp, clique) yields the 32-bit
// fit word; words are staged in shared memory and written back as full 128-byte lines per row.
// The same pass leaves the per-domain sum / max of the capacity bytes (non-unit levels): nodes are in topology order, so the
// lanes of a warp that share a domain are found once per level (__match_any_sync) and every (signature, level) costs the warp
// two reductions and a couple of atomics -- "sum over the fill domain >= MinReplicas" is the necessary condition K3's
// pre-filters test, so domains failing it are skipped without changing any result.
// ------------------------------------------------------------------------------------------------
constexpr int kFitTile = 4;     // signatures per CTA: the grid is (node tiles) x (signature tiles), every tile a short loop

// min(x / d, 256) for d > 0, exactly, without the ~20-instruction integer division: quotients that matter are small
// (a gang has at most GROVE_MAX_GANG_PODS pods; capacity bytes saturate at 255), so a float estimate is off by at most
// one and is corrected with one multiply
__device__ __forceinline__ uint32_t div_small(uint32_t x, uint32_t d) {
  if (x >= (uint64_t(d) << 8)) return 256u;
  uint32_t q = uint32_t(__fdividef(float(x), float(d)));   // x < 256 d: |error| <= 1
  if (uint64_t(q) * d > x) --q;
  if (x - q * d >= d) ++q;   // q d <= x now, so the difference does not wrap
  return q;
}

// K1 proper: fit(q, n) for every (signature, node) pair -> one bit; the same pass also leaves HOW MANY pods of the
// signature fit on the node (capacity byte, saturating at 255; fit <=> byte != 0), which K3 packs from.
__global__ void __launch_bounds__(1024) k_fit(Topo tp, Tables tb, uint32_t* __restrict__ F, uint8_t* __restrict__ cap8,
                                              uint32_t* capsum, uint32_t* capmax) {
  __shared__ uint4 s_prm[kFitTile];
  __shared__ uint32_t s_out[kFitTile][32];
  const uint32_t n_rows = tb.S;                            // every signature of the submission
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t node = blockIdx.x * 1024 + tid;           // npad is a multiple of 1024
  pdl_begin();
  const uint4 r = __ldg(tp.nres + node);
  const uint4 dm = __ldg(tp.ndom + node);
  const uint32_t gpu = r.z & 0xFFFFu, pods = r.z >> 16;
  const uint32_t depth = (r.w >> 16) & 0xFu;
  const uint32_t onehot = ((r.w & GROVE_NODE_SCHEDULABLE) && pods >= 1) ? (1u << ((r.w >> GROVE_NODE_CLASS_SHIFT) & 0xFu)) : 0u;
  // the lanes that share this node's domain, per non-unit level (capsum / capmax columns exist for those only)
  const uint32_t key[GROVE_MAX_LEVELS] = {dm.x, dm.y, dm.z, dm.w};
  uint32_t seg[GROVE_MAX_LEVELS], col[GROVE_MAX_LEVELS];
#pragma unroll
  for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) {
    seg[l] = 0; col[l] = GROVE_NONE_U32;
    if (l < tp.L && !tp.unit[l] && capsum) {
      seg[l] = __match_any_sync(kFull, key[l]);
      if (key[l] != GROVE_DOM_ABSENT && lane == uint32_t(__ffs(seg[l]) - 1)) col[l] = tp.cap_off[l] + key[l];   // the segment's first lane publishes
    }
  }
  for (uint32_t r0 = blockIdx.y * kFitTile; r0 < n_rows; r0 += gridDim.y * kFitTile) {
    __syncthreads();
    if (tid < kFitTile) s_prm[tid] = r0 + tid < n_rows ? tb.sigs[r0 + tid] : make_uint4(kFull, kFull, kFull, 0);  // never fits
    __syncthreads();
    const int cnt = int(min(uint32_t(kFitTile), n_rows - r0));
    for (int c = 0; c < cnt; ++c) {
      const uint4 p = s_prm[c];
      const bool ok = (r.x >= p.x) & (r.y >= p.y) & (gpu >= p.z) & ((p.w & onehot) != 0) & (depth >= (p.w >> 16));
      const uint32_t b = __ballot_sync(kFull, ok);
      if (lane == 0) s_out[c][warp] = b;
      uint32_t cap = 0;
      if (ok) {
        cap = pods;
        if (p.x) cap = min(cap, div_small(r.x, p.x));
        if (p.y) cap = min(cap, div_small(r.y, p.y));
        if (p.z) cap = min(cap, div_small(gpu, p.z));
        cap = min(cap, 255u);
      }
      cap8[size_t(r0 + c) * tp.npad + node] = uint8_t(cap);
      if (b) {   // (a warp without a fit node adds nothing: the tables were zeroed)
#pragma unroll
        for (uint32_t l = 0; l < GROVE_MAX_LEVELS; ++l) {
          if (seg[l]) {
            const uint32_t sum = __reduce_add_sync(seg[l], cap), mx = __reduce_max_sync(seg[l], cap);
            if (col[l] != GROVE_NONE_U32 && sum) {
              atomicAdd(capsum + size_t(r0 + c) * tp.cap_stride + col[l], sum);
              atomicMax(capmax + size_t(r0 + c) * tp.cap_stride + col[l], mx);
            }
          }
        }
      }
    }
    __syncthreads();
    for (int c = warp; c < cnt; c += 32) F[size_t(r0 + c) * tp.words + blockIdx.x * 32 + lane] = s_out[c][lane];
  }
}

}  // namespace grove
