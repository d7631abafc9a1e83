// sm_100a search kernels for the dense byte-class DFA tables produced by
// dfa/determinize.cpp.  Everything here is integer/byte work bound by HBM reads
// of the haystack and by shared-memory table lookups; there is no contraction,
// so no tensor cores (BASELINE.json north_star).
//
// Kernel inventory (reference function each replaces):
//   scan_rev_fast     all match STARTS of the haystack as a bitmap -- the chunk-parallel
//                     form of running exec_at_reverse (src/dfa.rs:768-866) from every
//                     match end -- on the shared-memory hot table, fed by 2-D tiled TMA;
//                     FUSED: each lane also walks the find_iter chain of its segment
//   scan_rev_bitmap   the same for tables that do not fit / special cases (generic)
//   scan_fwd_fast,    first match END / any match / RegexSet mask over one big
//   scan_fwd_reduce   haystack -- exec_at with quit_after_match (src/dfa.rs:576-764)
//                     and forward_many (:525-570)
//   walk_chunks,      the find_iter chain (src/re_trait.rs:197-220) over the start
//   stitch_check,     bitmap + anchored leftmost-first runs (exec_at); speculative per
//   compact_spans     chunk, validated against the left neighbour, ordered compaction
//   batch_fast,       one thread per record: is_match / find / set matches, the
//   *_batch           reference algorithm verbatim per record (exec.rs:632-662)
//   batch_refill      batched is_match with a warp's lanes refilled from a task of records
//   batch_iter*       one thread per record: find_iter (re_trait.rs:197-220) per record,
//                     count pass + prefix sum + write pass (CSR output)
//   batch_cand        batched records from candidate starts (over-budget patterns)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace rbgpu {

constexpr uint64_t kNone = ~0ull;        // "no position"
constexpr uint64_t kSpec = ~0ull - 1;    // chunk entry state is speculative
constexpr uint64_t kTooLong = ~0ull - 2; // an anchored run of a speculative chunk walk was cut off (see kSpecRunCap)
constexpr uint64_t kPending = ~0ull - 3; // a run longer than kTripRunCap inside a voting walk: taken up again after the trip loop
// Walks whose lanes vote once per trip (chunk_walk_simple / _lean) must not run a long match inside a
// trip: the vote is a barrier, so the other lanes would wait, and long runs that come up in different
// trips would execute one after the other (ncu: one thread per instruction, 0.2 s for 200 chunks).
// A run that passes this many bytes is left pending; all pending runs of a warp then go together.
constexpr uint64_t kTripRunCap = 2048;
// A speculatively entered chunk gives up on a match longer than this: with `(?s)foo.*bar` every
// chunk that holds a `foo` would otherwise run its automaton to the last `bar` of the haystack,
// only to learn from the stitch that the one real match covers it.  The chunk is DEFERRED instead:
// the stitch walks it again with its exact entry state (no cap) unless it is covered.
constexpr uint64_t kSpecRunCap = 1ull << 16;
// A chunk walked from its exact entry state hands a match longer than this to the host, which
// measures it with a parallel forward scan (engine.cu resolve_long_run) instead of one thread.
constexpr uint64_t kExactRunCap = 1ull << 18;
// Deferred chunks are walked again only within this many chunks of the leftmost deferred one: the
// chunks behind a long match are usually covered by it, and each walk costs up to a whole cap.
constexpr uint32_t kDeferredWindow = 1024;

struct DfaView {
  const uint16_t* trans;    // [n_states][stride], class-indexed; column stride-1 is EOF
  const uint8_t* classes;   // [256]
  const uint64_t* masks;    // [n_states][mask_words]
  uint32_t n_states, stride, match_lo, mask_words;
  uint32_t table_bytes;     // n_states * stride * 2
  uint16_t start[128];
  uint8_t uniform_start;
};

// Byte-indexed table over the HOT states of a DFA for the shared-memory fast kernels:
// either every state (small automata) or the states reachable from the start states
// through ASCII bytes only (Unicode-aware classes compile to hundreds of states of
// which an ASCII haystack visits a handful).  Hot ids: 0 = dead, 1 = trap (the
// transition left the hot set; absorbing), then non-match states, then match states.
// A lane that lands in the trap row re-runs those bytes on the full class-indexed table.
#ifndef RB_HOT_ROW
#define RB_HOT_ROW 280  // bytes between hot-table rows in shared memory: 256 entries + 24 (rows start 6 banks apart; tools/micro/bank_sim.py)
#endif
struct HotView {
  const uint16_t* next256;   // [n][256] successor hot ids
  const uint16_t* eof;       // [n] EOF successor in FULL numbering
  const uint16_t* hot2full;  // [n]
  const uint16_t* full2hot;  // [full n_states], 0xFFFF = cold
  uint32_t n, match_lo;      // rows; hot ids >= match_lo are match states
  uint32_t start;            // hot id of the uniform start state (forward runner)
};

__device__ __forceinline__ bool is_word_byte(uint32_t b) {
  return (b - 'a' < 26u) || (b - 'A' < 26u) || (b - '0' < 10u) || b == '_';
}

// dfa.rs:1415-1434 / 1440-1464 (flag index layout: determinize.h)
__device__ __forceinline__ int flags_forward(const uint8_t* t, uint64_t n, uint64_t at) {
  int f = 0;
  if (at == 0) f |= 1;
  if (n == 0) f |= 2 | 8;
  if (at == 0 || t[at - 1] == '\n') f |= 4;
  bool last = at > 0 && is_word_byte(t[at - 1]);
  bool cur = at < n && is_word_byte(t[at]);
  f |= (last == cur) ? 32 : 16;
  if (last) f |= 64;
  return f;
}
__device__ __forceinline__ int flags_reverse(const uint8_t* t, uint64_t n, uint64_t at) {
  int f = 0;
  if (at == n) f |= 1;
  if (n == 0) f |= 2 | 8;
  if (at == n || t[at] == '\n') f |= 4;
  bool last = at < n && is_word_byte(t[at]);
  bool cur = at > 0 && is_word_byte(t[at - 1]);
  f |= (last == cur) ? 32 : 16;
  if (last) f |= 64;
  return f;
}

// A DFA whose table (and class map) may have been staged into shared memory.
struct Table {
  const uint16_t* trans;
  const uint8_t* classes;
  uint32_t stride;
  __device__ __forceinline__ uint32_t step(uint32_t s, uint32_t byte) const {
    return trans[s * stride + classes[byte]];
  }
  __device__ __forceinline__ uint32_t step_eof(uint32_t s) const { return trans[s * stride + stride - 1]; }
};

// Cooperative copy of table + class map into dynamic shared memory when it fits.
__device__ __forceinline__ Table stage_table(const DfaView& d, unsigned char* smem, bool use_smem) {
  Table t;
  t.stride = d.stride;
  if (use_smem) {
    uint16_t* st = reinterpret_cast<uint16_t*>(smem);
    uint8_t* sc = smem + ((d.table_bytes + 15) & ~15u);
    const uint32_t n16 = d.table_bytes / 2;
    for (uint32_t i = threadIdx.x; i < n16; i += blockDim.x) st[i] = d.trans[i];
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) sc[i] = d.classes[i];
    __syncthreads();
    t.trans = st;
    t.classes = sc;
  } else {
    t.trans = d.trans;
    t.classes = d.classes;
  }
  return t;
}
// The table and class map where the view keeps them (global memory).
__device__ __forceinline__ Table global_table(const DfaView& d) { return Table{d.trans, d.classes, d.stride}; }

}  // namespace rbgpu
