// common.cuh -- shared structs of the placement kernels (device views of the tables, relaxation state).
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/grove_place.h"


namespace grove {

constexpr uint32_t kFull = 0xFFFFFFFFu;
constexpr int kMaxPieces = 2 * GROVE_MAX_LEVELS + 3;
constexpr uint32_t kClaimSlots = 8;           // inline claim slots per node (one 128 B line); more spill to the overflow list
constexpr uint32_t kClaimEmpty = 0xFFFFFFFFu;
constexpr uint32_t kStale = 0x80u;            // nlive8 bit: committed state changed since the capacity tables were built
constexpr uint32_t kHasOvf = 0x40u;           // nlive8 bit: the node has (had) claims in the overflow chain
constexpr uint32_t kTagRounds = 254u;         // rounds per stamp epoch (stamps carry a round tag in their top byte)

struct GangInfo {     // 48 B, built on the host at submit time
  uint32_t anchor;    // sorted node index
  uint32_t order;     // rank by (priority desc, index asc)
  uint32_t pod_off;   // first slot in the entry arrays
  uint32_t pad;       // gang shape id (gangs with identical structure share one candidate pre-filter row)
  uint32_t anc_lo[GROVE_MAX_LEVELS];  // node range of the anchor's domain per level; [a,a) if label absent
  uint32_t anc_hi[GROVE_MAX_LEVELS];
};

struct CliqueInfo {   // 16 B
  uint32_t gang;
  uint32_t need_depth;  // labels a candidate node must carry (deepest binding Required level + 1)
  uint32_t sig;         // fit signature: cliques with identical (requests, class mask, need_depth) share a fit row
  uint32_t pad;
};

struct Topo {
  const uint4* nres;       // [npad] committed state: free_cpu, free_mem, free_gpu | free_pods << 16, flags | vdepth << 16
  const uint4* ndom;       // [npad] static: tree-ified domain index per level
  const uint32_t* dom_lo[GROVE_MAX_LEVELS];
  const uint32_t* dom_hi[GROVE_MAX_LEVELS];
  const uint32_t* next_dom[GROVE_MAX_LEVELS];  // [n+1] first level-l domain starting at or after node i
  uint32_t n_dom[GROVE_MAX_LEVELS];
  uint32_t unit[GROVE_MAX_LEVELS];             // every domain of the level is a single node
  uint32_t n, npad, L, words;                  // words = npad / 32 (row stride of the fit bitmap)
  uint32_t cap_off[GROVE_MAX_LEVELS];          // column offset of level l in a capacity-table row (non-unit levels)
  uint32_t cap_stride;                         // columns per signature row = sum of n_dom over non-unit levels
};

struct Tables {
  const grove_gang_t* gangs;
  const grove_clique_t* cliques;
  const grove_scope_t* scopes;
  const GangInfo* ginfo;
  const CliqueInfo* cinfo;
  const uint4* sigs;        // [S] req_cpu, req_mem, req_gpu, class_mask | need_depth << 16
  const uint32_t* by_rank;  // [G] gang index at each order rank
  uint32_t G, Q, S, NS;     // NS = scopes in the submission
};

// Control words of the relaxation (device memory; the host reads them back once per round or not at all)
enum Ctl : uint32_t {
  kFront = 0,      // settled prefix: every gang of rank < front is final
  kHi,             // window end: gangs of rank in [front, hi) relax
  kRound,          // relaxation round, from 1
  kNEval,          // gangs evaluated this round: the list (heavy + light) and the new entrants
  kMinDirty,       // lowest rank that has to be (re-)evaluated after this round (becomes the next front)
  kChanged,        // gangs whose tentative result changed this round
  kEvals,          // evaluations so far (stat)
  kOvfCount,       // entries handed out of the claim overflow pool
  kRemAny,         // stamp (tag | rank): lowest rank that withdrew a claim this round
  kDone,           // 1 when front == G
  kTablesAt,       // front at the last capacity-table build
  kRefresh,        // 1: rebuild the capacity tables before the next evaluation
  kCtaDone,        // last-CTA-done counter of k_detect
  kFoldAny,        // (unused)
  kNHeavy,         // gangs at the head / tail of eval_list (written by k_detect of the round before)
  kNLight,
  kFolded,         // ranks below this are folded into the committed state (k_fold): folded <= front
  kEntryLo,        // this round's new entrants are the ranks [kEntryLo, kHi): never evaluated, no list entry needed
  kNHeavyNext,     // the NEXT round's list counters, filled by k_detect while this round's are still being read
  kNLightNext,
  kCtlWords = 24
};

// Progress words in host-mapped memory, written by the last CTA of k_detect after every round (kLiveRound last, behind a
// system-wide fence): the host learns that a round is over, whether the cycle is, and whether a table rebuild is due, by
// reading memory -- no blocking call, no idle GPU between batches of rounds.
enum Live : uint32_t { kLiveRound = 0, kLiveFront, kLiveDone, kLiveRefresh, kLiveOvf, kLiveEvals, kLiveWords = 8 };

// Relaxation state.  A gang's tentative result ("cur") lives in its own slots of the entry arrays and becomes final
// in place; "nxt" is the scratch an evaluation writes before k_apply compares and publishes it.
struct Relax {
  uint32_t* ctl;            // [kCtlWords]
  uint8_t* state;           // [G] final GROVE_GANG_* (PENDING until settled)
  uint8_t* tstate;          // [G] tentative state of the last evaluation (0 = never evaluated)
  uint8_t* dirty;           // [G] must be re-evaluated next round
  uint32_t* chg_round;      // [G] last round in which the gang's tentative result changed
  uint32_t* eval_list;      // [G] the gangs to re-evaluate: heavy ones from the head, light ones from the tail (k_detect)
  uint8_t* last_att;        // [G] attempt rounds the gang's last evaluation needed
  // tentative / final result per gang
  uint32_t* ent_node;       // [P]
  uint16_t* ent_meta;       // [P] clique_rel
  uint16_t* cur_n;          // [G] entries incl. surplus
  uint32_t* cur_info;       // [G] gang level got (0xFF none) | score_num << 8 | score_den << 20
  uint32_t* cur_glo;        // [G] first sorted node of the gang domain
  uint32_t* extent;         // [G] nodes of the gang's visiting order its last evaluation may have read
  uint8_t* sc_lvl;          // [NS] level each scope was packed at (0xFF: no own domain)
  uint32_t* sc_lo;          // [NS]
  // scratch of this round's evaluations
  uint32_t* nxt_node;       // [P]
  uint16_t* nxt_meta;       // [P]
  uint16_t* nxt_n;          // [G]
  uint8_t* nxt_tstate;      // [G]
  uint32_t* nxt_info;       // [G]
  uint32_t* nxt_glo;        // [G]
  uint32_t* nxt_extent;     // [G]
  uint8_t* nxt_sc_lvl;      // [NS]
  uint32_t* nxt_sc_lo;      // [NS]
  // claims of the tentative results: what gangs of higher rank subtract from the committed state
  uint4* claims;            // [npad][kClaimSlots] x = rank (kClaimEmpty = free), y = cpu, z = mem, w = gpu | pods << 16
  uint32_t* nlive;          // [npad / 4] one byte per node: live inline claims | kHasOvf | kStale
  uint32_t* ovf_head;       // [npad] first entry + 1 of the node's overflow chain (0 = none)
  uint32_t* ovf_next;       // [ovf_cap] next entry + 1
  uint4* ovf_claim;         // [ovf_cap] same layout as a claim slot; dead entries (x = kClaimEmpty) are revived by later claims on the node
  uint32_t ovf_cap;
  int4* ctot;               // [npad] sum of ALL live claims on the node (inline + overflow): cpu, mem, gpu, pods
  uint32_t* cmaxr;          // [npad] upper bound of the ranks that claim(ed) the node this cycle: a gang of a higher rank sees
                            // committed - ctot and never reads the claim line
  // change stamps of the round: (tag << 24) | lowest rank; a stale tag = no stamp
  uint32_t* add_stamp;      // [npad] a gang newly claimed this node
  uint32_t* rem_stamp;      // [words] a gang withdrew a claim from this 32-node group
  uint32_t* rem_round;      // [words] last round in which ANY gang withdrew a claim from the group
  uint32_t* last_eval;      // [G] round of the gang's last evaluation (0 = never)
  uint32_t* fail_upto;      // [G] candidates (in order) that came before the last evaluation's answer: all of them failed then
  // capacity tables over the committed state as of the last build (upper bounds afterwards)
  uint32_t* F;              // [S][words] fit bitmap, one row per signature
  uint8_t* cap8;            // [S][npad] pods of the signature that fit on the node (saturating at 255)
  uint32_t* capsum;         // [S][cap_stride] per-domain sum of cap8 (non-unit levels)
  uint32_t* capmax;         // [S][cap_stride] per-domain max of cap8
  uint8_t* T;               // [Q][npad] K2 score matrix over the cycle-start snapshot
  const uint32_t* shape_bits; // [shapes][pl_words] candidate pre-filter per (gang shape, domain), bit pl_off[level] + d; null = not built
  uint32_t pl_off[GROVE_MAX_LEVELS], pl_words;
  uint32_t P, window, entry, heavy_att;   // heavy_att: attempts of its last evaluation from which a gang counts as heavy
  uint32_t* dbg;            // [G][8] optional per-gang evaluation statistics
  uint32_t* live;           // [kLiveWords] host-mapped: progress words the host polls (null: not available)
};

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, uint32_t lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(kFull, v, d);
    if (lane >= (uint32_t)d) v += t;
  }
  return v;
}

// stamp of round r for rank k: newer rounds carry SMALLER tags, so atomicMin lets a newer stamp beat a stale one
__device__ __forceinline__ uint32_t stamp_tag(uint32_t round) { return kTagRounds - (round % kTagRounds); }  // 1..254
__device__ __forceinline__ uint32_t make_stamp(uint32_t round, uint32_t rank) { return (stamp_tag(round) << 24) | rank; }
__device__ __forceinline__ bool stamp_below(uint32_t s, uint32_t round, uint32_t rank) {
  return (s >> 24) == stamp_tag(round) && (s & 0xFFFFFFu) < rank;
}

// Programmatic dependent launch: the kernels of a cycle after k_reset are launched so that the next one's CTAs can be
// resident before this one ends (engine.cu launch_pdl).  Every such kernel calls pdl_begin() before its first global load,
// store or atomic: griddepcontrol.wait returns once the preceding grid has completed and its writes are visible (at once
// when the preceding operation was not a dependent launch), so ordering stays transitive along the stream; the trigger
// right after it lets the next kernel be scheduled.
__device__ __forceinline__ void pdl_begin() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

}  // namespace grove
