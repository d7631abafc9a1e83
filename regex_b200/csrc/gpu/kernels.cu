// Kernel definitions; see kernels.cuh for the inventory and engine.cu for launches.
#include <cuda.h>

#include "kernels.cuh"
#include <type_traits>
#include "launch.h"

namespace rbgpu {

extern __shared__ __align__(16) unsigned char g_smem[];

__device__ __forceinline__ uint4 ldg128(const uint8_t* p);
__device__ __forceinline__ uint32_t word_byte(const uint4& v, int j) {  // byte j (0..15) of a 16-byte vector
  const uint32_t w = (j >> 2) == 0 ? v.x : (j >> 2) == 1 ? v.y : (j >> 2) == 2 ? v.z : v.w;
  return (w >> (8 * (j & 3))) & 0xFFu;
}
// one whole 32-byte sector {w0 (lowest address), w1, w2, w3}; p is 32-byte aligned
__device__ __forceinline__ void st_sector(uint64_t* p, uint64_t w0, uint64_t w1, uint64_t w2, uint64_t w3) {
  asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(w0), "l"(w1), "l"(w2), "l"(w3) : "memory");
}
__device__ __forceinline__ uint32_t pick_start_rev(const DfaView& d, const uint8_t* t, uint64_t n, uint64_t at) {
  return d.uniform_start ? d.start[32] : d.start[flags_reverse(t, n, at)];
}
__device__ __forceinline__ uint32_t pick_start_fwd(const DfaView& d, const uint8_t* t, uint64_t n, uint64_t at) {
  return d.uniform_start ? d.start[32] : d.start[flags_forward(t, n, at)];
}

// ------------------------------------------------------------ scan_rev_bitmap --
// Bitmap format: bit i is set iff a match STARTS at position i+1, i.e. iff the
// reverse automaton reports a (delayed) match when it consumes text[i].  A match
// starting at position 0 is reported by the EOF step into *flag0.
// Segment t owns bytes [base + t*seg, base + (t+1)*seg) ∩ [0, n).  The state at
// the top of a segment is guessed by running the automaton from a fresh start
// state `warm` bytes further right; verify_segments() checks every guess
// against the neighbour's exact final state and lists the segments to redo.
//
// Generic version: any table size (shared memory when it fits, else L1/L2), any
// alignment, optional UTF-8 boundary mask.  Two lookups per byte; the haystack is read
// with 16-byte loads when the buffer is 16-byte aligned (a byte load per lane costs the
// warp 32 L1 wavefronts per byte-step, a 16-byte load 32 per sixteen).
__global__ void scan_rev_bitmap(ScanArgs a) {
  const Table T = stage_table(a.dfa, g_smem, a.use_smem);
  const bool vec = (reinterpret_cast<uintptr_t>(a.text) & 15) == 0;
  const uint64_t total = a.redo_list ? (uint64_t)*a.n_redo : a.n_seg;
  const uint32_t match_lo = a.dfa.match_lo;
  for (uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t t = a.redo_list ? a.redo_list[idx] : idx;
    const uint64_t lo = min(a.base + t * a.seg, a.limit);
    const uint64_t hi = min(lo + a.seg, a.limit);  // bytes [lo, hi); limit <= n (shards scan their own bytes only)
    uint32_t s;
    if (a.redo_list) {
      s = a.fin[t + 1];
    } else {
      const uint64_t w = min(hi + a.warm, a.n);
      s = pick_start_rev(a.dfa, a.text, a.n, w);
      uint64_t i = w;
      while (i > hi && (!vec || (i & 15) || i - hi < 16)) { i--; s = T.step(s, a.text[i]); }
      while (i > hi) {  // vec: i and hi are 16-byte aligned here
        const uint4 v = ldg128(a.text + i - 16);
#pragma unroll
        for (int j = 15; j >= 0; j--) s = T.step(s, word_byte(v, j));
        i -= 16;
      }
    }
    a.guess[t] = (uint16_t)s;
    uint64_t word = 0;
    uint32_t next_byte = hi < a.n ? a.text[hi] : 0;  // text[i+1], for the UTF-8 boundary mask
    auto consume = [&](uint32_t b, uint64_t pos) {
      s = T.step(s, b);
      bool hit = s >= match_lo;
      if (a.utf8_boundaries && (next_byte & 0xC0) == 0x80) hit = false;
      if (hit) word |= 1ull << (pos & 63);
      next_byte = b;
      if ((pos & 63) == 0 || pos == lo) { a.bitmap[pos >> 6] = word; word = 0; }
    };
    uint64_t i = hi;
    while (i > lo && (!vec || (i & 15) || i - lo < 16)) { i--; consume(a.text[i], i); }
    while (i > lo) {  // vec: 16-byte aligned, lo is a multiple of 64
      const uint4 v = ldg128(a.text + i - 16);
#pragma unroll
      for (int j = 15; j >= 0; j--) consume(word_byte(v, j), i - 16 + j);
      i -= 16;
    }
    a.fin[t] = (uint16_t)s;
    if (lo == 0) {
      bool hit0 = T.step_eof(s) >= match_lo;
      if (a.utf8_boundaries && (next_byte & 0xC0) == 0x80 && a.n > 0) hit0 = false;
      *a.flag0 = hit0;
    }
  }
}

// Fast version for hot tables (kernels.cuh HotView) staged in shared memory:
//   - ONE-BYTE entries: row r holds the 256 successor ids of hot state r, rows are
//     kHotRow = 288 bytes apart.  With 4-byte entries a row covers all 32 banks, so lanes
//     in different states collide at random (ncu: 2.1 wavefronts per look-up, the
//     kernel's binding cost).  With one-byte entries the letters a-z of one row live in 7
//     consecutive words, and the 32 spare bytes per row start consecutive rows 8 banks
//     apart: the few states a text automaton spends its time in use disjoint banks, and
//     lanes reading neighbouring bytes of one row share a word (broadcast).
//   - a step is PRMT (haystack byte k merged into the 256-aligned table address) +
//     IMAD (state * 288 + that) + LDS.U8; the state IS the row index, match rows sit
//     above non-match rows ("e >= match_lo"), row 0 = dead, row 1 = trap.
//   - bits are assembled in registers, one 64-bit store per 64 bytes of text.
constexpr uint32_t kHotRow = RB_HOT_ROW;
__device__ __forceinline__ uint32_t hot_table_bytes(uint32_t rows) { return (rows * kHotRow + 255u) & ~255u; }
__device__ __forceinline__ uint32_t lds8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// successor of state e on byte K (compile-time) of the little-endian word w; tb = 256-aligned table address
template <int K>
__device__ __forceinline__ uint32_t hot_next(uint32_t tb, uint32_t w, uint32_t e) {
  const uint32_t x = __byte_perm(w, tb, 0x7650 + K);  // tb | byte K of w
  uint32_t addr;
  asm("mad.lo.u32 %0, %1, %3, %2;" : "=r"(addr) : "r"(e), "r"(x), "n"(RB_HOT_ROW));
  return lds8(addr);
}
__device__ __forceinline__ uint32_t hot_next_b(uint32_t tb, uint32_t byte, uint32_t e) { return lds8(tb + e * kHotRow + byte); }
// cooperative expansion of a hot table into shared memory (4 entries per store)
__device__ __forceinline__ void hot_stage(const HotView& h, uint32_t tb) {
  const uint32_t n4 = h.n * 64u;
  const uint2* src = reinterpret_cast<const uint2*>(h.next256);  // 4 x u16
  for (uint32_t i = threadIdx.x; i < n4; i += blockDim.x) {
    const uint2 v = src[i];
    const uint32_t packed = (v.x & 0xFFu) | ((v.x >> 8) & 0xFF00u) | ((v.y & 0xFFu) << 16) | ((v.y >> 16) << 24);
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(tb + (i >> 6) * kHotRow + (i & 63u) * 4u), "r"(packed));
  }
}
__device__ __forceinline__ uint4 ldg128(const uint8_t* p) {
  uint4 v;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
// Consume the 4 bytes of w from the highest address down; BIT0 = bit index of byte 0.
template <int BIT0>
__device__ __forceinline__ void rev_word(uint32_t tb, uint32_t w, uint32_t& e, uint32_t& bits, uint32_t thr) {
  e = hot_next<3>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 3);
  e = hot_next<2>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 2);
  e = hot_next<1>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 1);
  e = hot_next<0>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 0);
}
template <int BIT0>
__device__ __forceinline__ void rev_block16(uint32_t tb, const uint4& v, uint32_t& e, uint32_t& bits, uint32_t thr) {
  rev_word<BIT0 + 12>(tb, v.w, e, bits, thr);
  rev_word<BIT0 + 8>(tb, v.z, e, bits, thr);
  rev_word<BIT0 + 4>(tb, v.y, e, bits, thr);
  rev_word<BIT0 + 0>(tb, v.x, e, bits, thr);
}

// ---- signed row ids (scan_rev_fast's own table) ----
// The reverse scan records one bit per byte: "did this step enter a match state".  With row
// ids 0..n-1 that is a compare plus a predicated add per byte (ISETP + @P VIADD).  Here match
// rows get NEGATIVE ids -1, -2, ... and live BELOW the table's base address (the row address
// is still base + id * 288, two's complement), entries are loaded sign-extended (LDS.S8), and
// the bit is the sign: bits = funnel_shift_left(id, bits, 1) -- ONE instruction.  A byte then
// costs PRMT + IMAD + LDS.S8 + SHF instead of five instructions.  Non-match rows keep ids
// 0 (dead), 1 (trap), 2...; at most 128 of either kind.
__device__ __forceinline__ uint32_t hot_signed_below(const HotView& h) { return ((h.n - h.match_lo) * kHotRow + 255u) & ~255u; }  // bytes of match rows
__device__ __forceinline__ uint32_t hot_signed_bytes(const HotView& h) { return hot_signed_below(h) + ((h.match_lo * kHotRow + 255u) & ~255u); }
__device__ __forceinline__ uint32_t hot_sid(uint32_t idx, uint32_t match_lo) { return idx < match_lo ? idx : ~(idx - match_lo); }   // row index -> signed id
__device__ __forceinline__ uint32_t hot_idx(uint32_t sid, uint32_t match_lo) { return (int32_t)sid >= 0 ? sid : match_lo + ~sid; } // and back
__device__ __forceinline__ void hot_stage_signed(const HotView& h, uint32_t mid) {  // mid = address of row 0 (256-byte aligned)
  const uint32_t n4 = h.n * 64u;
  const uint2* src = reinterpret_cast<const uint2*>(h.next256);  // 4 x u16 row indices
  const uint32_t ml = h.match_lo;
  for (uint32_t i = threadIdx.x; i < n4; i += blockDim.x) {
    const uint2 v = src[i];
    const uint32_t a = hot_sid(v.x & 0xFFFFu, ml) & 0xFFu, b = hot_sid(v.x >> 16, ml) & 0xFFu;
    const uint32_t c = hot_sid(v.y & 0xFFFFu, ml) & 0xFFu, d = hot_sid(v.y >> 16, ml) & 0xFFu;
    const uint32_t row = (uint32_t)((int32_t)mid + (int32_t)hot_sid(i >> 6, ml) * (int32_t)kHotRow);
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(row + (i & 63u) * 4u), "r"(a | (b << 8) | (c << 16) | (d << 24)));
  }
}
template <int K>
__device__ __forceinline__ uint32_t hot_next_s(uint32_t mid, uint32_t w, uint32_t e) {
  const uint32_t x = __byte_perm(w, mid, 0x7650 + K);  // mid | byte K of w
  uint32_t addr, v;
  asm("mad.lo.u32 %0, %1, %3, %2;" : "=r"(addr) : "r"(e), "r"(x), "n"(RB_HOT_ROW));
  asm volatile("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// Consume the 4 bytes of w from the highest address down; after 32 such steps bit i of `bits` is byte i.
__device__ __forceinline__ void rev_word_s(uint32_t mid, uint32_t w, uint32_t& e, uint32_t& bits) {
  e = hot_next_s<3>(mid, w, e); bits = __funnelshift_l(e, bits, 1);
  e = hot_next_s<2>(mid, w, e); bits = __funnelshift_l(e, bits, 1);
  e = hot_next_s<1>(mid, w, e); bits = __funnelshift_l(e, bits, 1);
  e = hot_next_s<0>(mid, w, e); bits = __funnelshift_l(e, bits, 1);
}
__device__ __forceinline__ void rev_block16_s(uint32_t mid, const uint4& v, uint32_t& e, uint32_t& bits) {
  rev_word_s(mid, v.w, e, bits);
  rev_word_s(mid, v.z, e, bits);
  rev_word_s(mid, v.y, e, bits);
  rev_word_s(mid, v.x, e, bits);
}

// ---- TMA ring: per-lane 64-byte groups land in shared memory through cp.async.bulk ----
// Uncoalesced per-lane LDG.128 costs one L1TEX wavefront per lane (ncu: L1/TEX at 98 %
// with half of it global loads).  Bulk copies bypass the LSU path; each lane then
// reads its own 64 bytes with four LDS.128 (conflict-free in the 2-D TMA layout below).
constexpr uint32_t kRingLaneStride = 64;                       // one 64-byte group per lane
constexpr uint32_t kRingStageBytes = 32 * kRingLaneStride;     // per warp
constexpr uint32_t kBoxStages = 2;                             // ring depth (3 measured slower: 2.15 -> 2.59 ms on 4 GiB, less L1 left)
constexpr uint32_t kRingWarpBytes = kBoxStages * kRingStageBytes;  // 512-byte aligned (TMA 64B-swizzle pattern)
constexpr uint32_t kRingBarBytes = 64;                         // 2 + kBoxStages 8-byte mbarriers per warp, after all rings

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@!p bra W;\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// One 2-D tiled TMA load: a [16 B x 32 rows] box (one 16-byte piece of 32 consecutive
// segments) lands as 512 contiguous bytes, so lane j finds its piece at +16*j.
__device__ __forceinline__ void tma_box(uint32_t dst, const CUtensorMap* map, uint32_t col, uint32_t row, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(map), "r"(col), "r"(row), "r"(bar) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// ------------------------------------------------------------ scan_fwd_reduce --
// Mirror image for forward all-match scans.  Position q is a match END iff the
// automaton, standing at q, reports a match when it consumes text[q] (EOF at n).
// Per segment: the first match end and the OR of the per-state pattern masks.
__global__ void scan_fwd_reduce(ScanArgs a) {
  const Table T = stage_table(a.dfa, g_smem, a.use_smem);
  const bool vec = (reinterpret_cast<uintptr_t>(a.text) & 15) == 0;
  const uint64_t total = a.redo_list ? (uint64_t)*a.n_redo : a.n_seg;
  const uint32_t match_lo = a.dfa.match_lo, mw = a.dfa.mask_words;
  for (uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t t = a.redo_list ? a.redo_list[idx] : idx;
    if (!a.redo_list && t >= a.skip_lo && t < a.skip_hi) continue;  // scan_fwd_fast's share
    const uint64_t lo = a.base + t * a.seg;
    const uint64_t hi = min(lo + a.seg, a.fwd_limit);
    uint32_t s;
    if (a.redo_list) {
      s = a.fin[t - 1];
    } else if (t == 0 && a.entry0 != kNoEntry) {
      s = a.entry0;
    } else {
      const uint64_t w = (lo - a.base > a.warm) ? lo - a.warm : a.base;
      s = pick_start_fwd(a.dfa, a.text, a.n, w);
      uint64_t q = w;
      while (q < lo && (!vec || (q & 15) || lo - q < 16)) { s = T.step(s, a.text[q]); q++; }
      while (q < lo) {
        const uint4 v = ldg128(a.text + q);
#pragma unroll
        for (int j = 0; j < 16; j++) s = T.step(s, word_byte(v, j));
        q += 16;
      }
    }
    a.guess[t] = (uint16_t)s;
    uint64_t first = kNone;
    uint64_t acc[kMaxMaskWords] = {0, 0, 0, 0};
    uint32_t last_match = 0;  // masks of this state are already in acc
    auto consume = [&](uint32_t ns, uint64_t pos) {
      s = ns;
      if (s >= match_lo) {
        if (first == kNone) first = pos;
        if (a.seg_mask && s != last_match) {
          last_match = s;
#pragma unroll
          for (uint32_t w = 0; w < kMaxMaskWords; w++)
            if (w < mw) acc[w] |= a.dfa.masks[(uint64_t)s * mw + w];
        }
      }
    };
    uint64_t q = lo;
    const uint64_t text_hi = min(hi, a.n);  // bytes [lo, text_hi), then the EOF step if hi == n + 1
    while (q < text_hi && (!vec || (q & 15) || text_hi - q < 16)) { consume(T.step(s, a.text[q]), q); q++; }
    while (q + 16 <= text_hi) {
      const uint4 v = ldg128(a.text + q);
#pragma unroll
      for (int j = 0; j < 16; j++) consume(T.step(s, word_byte(v, j)), q + j);
      q += 16;
    }
    while (q < text_hi) { consume(T.step(s, a.text[q]), q); q++; }
    if (q < hi) consume(T.step_eof(s), q);  // q == n, fwd_limit == n + 1
    a.fin[t] = (uint16_t)s;
    a.seg_first[t] = first;
    if (a.seg_mask) {
#pragma unroll
      for (uint32_t w = 0; w < kMaxMaskWords; w++)
        if (w < mw) a.seg_mask[t * mw + w] = acc[w];
    }
  }
}

// guess[t] must equal the exact state the neighbouring segment ended in.
__global__ void verify_segments(const uint16_t* guess, const uint16_t* fin, uint64_t n_seg, int reverse,
                                uint32_t* redo_list, uint32_t* n_redo) {
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < n_seg; t += (uint64_t)gridDim.x * blockDim.x) {
    bool bad;
    if (reverse) bad = t + 1 < n_seg && guess[t] != fin[t + 1];
    else bad = t > 0 && guess[t] != fin[t - 1];
    if (bad) redo_list[atomicAdd(n_redo, 1u)] = (uint32_t)t;
  }
}

// ---- exact entry states by state-map composition ------------------------------------
// The warm-up guess of a segment's entry state is wrong for automata whose state depends
// on far context (`(?s)foo.*bar`: "a bar lies somewhere to the right"), and redoing from
// the neighbour's state repairs only one more segment per round.  After a few rounds the
// engine switches to the north star's formulation: run every segment from EVERY state
// that occurs at a boundary (K, closed under the maps), compose the per-segment maps
// K -> K along the scan direction in three short kernels (blocks, block entries, fill),
// and redo once from the exact entry states.  Work: (|K| + 2) passes, no cascade.
__global__ void mark_states(const uint16_t* a, uint64_t n, uint8_t* present) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) present[a[i]] = 1;
}
__global__ void scan_map(ScanArgs a, int reverse, const uint16_t* states, uint32_t k, uint16_t* maps) {
  const Table T = stage_table(a.dfa, g_smem, a.use_smem);
  const uint64_t total = a.n_seg * k;
  for (uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; idx < total; idx += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t t = idx / k;  // the k threads of a segment are neighbours: their haystack loads coalesce into one
    uint32_t s = states[idx - t * k];
    const bool vec = (reinterpret_cast<uintptr_t>(a.text) & 15) == 0;
    if (reverse) {  // bytes [lo, hi) from the top down, as scan_rev_bitmap
      const uint64_t lo = min(a.base + t * a.seg, a.limit), hi = min(lo + a.seg, a.limit);
      uint64_t i = hi;
      while (i > lo && (!vec || (i & 15) || i - lo < 16)) { i--; s = T.step(s, a.text[i]); }
      while (i > lo) {  // i and lo are 16-byte aligned here
        const uint4 v = ldg128(a.text + i - 16);
#pragma unroll
        for (int j = 15; j >= 0; j--) s = T.step(s, word_byte(v, j));
        i -= 16;
      }
    } else {        // bytes [lo, hi) upwards, as scan_fwd_reduce (the EOF step belongs to no map)
      const uint64_t lo = a.base + t * a.seg, hi = min(lo + a.seg, a.n);
      uint64_t q = lo;
      while (q < hi && (!vec || (q & 15) || hi - q < 16)) { s = T.step(s, a.text[q]); q++; }
      while (q + 16 <= hi) {
        const uint4 v = ldg128(a.text + q);
#pragma unroll
        for (int j = 0; j < 16; j++) s = T.step(s, word_byte(v, j));
        q += 16;
      }
      while (q < hi) { s = T.step(s, a.text[q]); q++; }
    }
    maps[idx] = (uint16_t)s;
  }
}
__global__ void closure_check(const uint16_t* maps, uint64_t n, const uint16_t* kidx, uint8_t* present, uint32_t* n_new) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint16_t v = maps[i];
    if (kidx[v] == 0xFFFFu && !present[v]) { present[v] = 1; atomicAdd(n_new, 1u); }
  }
}
__global__ void compose_blocks(const uint16_t* maps, const uint16_t* kidx, const uint16_t* states, uint32_t k, uint64_t n_seg,
                               int reverse, uint16_t* comp) {
  const uint64_t n_blocks = (n_seg + kMapBlock - 1) / kMapBlock;
  const uint64_t id = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (id >= n_blocks * k) return;
  const uint64_t b = id / k;
  uint32_t s = states[id - b * k];
  const uint64_t t_lo = b * kMapBlock, t_hi = min(t_lo + kMapBlock, n_seg);
  if (reverse) for (uint64_t t = t_hi; t-- > t_lo;) s = maps[t * k + kidx[s]];
  else for (uint64_t t = t_lo; t < t_hi; t++) s = maps[t * k + kidx[s]];
  comp[id] = (uint16_t)s;
}
__global__ void compose_top(const uint16_t* comp, const uint16_t* kidx, uint32_t k, uint64_t n_blocks, int reverse,
                            const uint16_t* first_entry, uint16_t* block_entry) {
  if (blockIdx.x || threadIdx.x) return;
  uint32_t s = *first_entry;
  if (reverse) for (uint64_t b = n_blocks; b-- > 0;) { block_entry[b] = (uint16_t)s; s = comp[b * k + kidx[s]]; }
  else for (uint64_t b = 0; b < n_blocks; b++) { block_entry[b] = (uint16_t)s; s = comp[b * k + kidx[s]]; }
}
__global__ void compose_fill(const uint16_t* maps, const uint16_t* kidx, uint32_t k, uint64_t n_seg, int reverse,
                             const uint16_t* block_entry, uint16_t* exact) {
  const uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (b * kMapBlock >= n_seg) return;
  uint32_t s = block_entry[b];
  const uint64_t t_lo = b * kMapBlock, t_hi = min(t_lo + kMapBlock, n_seg);
  if (reverse) for (uint64_t t = t_hi; t-- > t_lo;) { exact[t] = (uint16_t)s; s = maps[t * k + kidx[s]]; }
  else for (uint64_t t = t_lo; t < t_hi; t++) { exact[t] = (uint16_t)s; s = maps[t * k + kidx[s]]; }
}
__global__ void publish_exact(const uint16_t* exact, uint64_t n_seg, int reverse, uint16_t* fin) {
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < n_seg; t += (uint64_t)gridDim.x * blockDim.x) {
    if (reverse) { if (t + 1 < n_seg) fin[t + 1] = exact[t]; }  // segment t enters with the final state of t + 1
    else if (t > 0) fin[t - 1] = exact[t];
  }
}

// One long anchored run, in parallel (engine.cu resolve_long_run): every segment is entered in its
// exact state (state-map composition), so "the last position at which the leftmost-first
// automaton was in a match state before it died" is a maximum over segments.
__global__ void scan_last_match(ScanArgs a, const uint16_t* exact, unsigned long long* best, uint32_t* alive_at_end) {
  const Table T = stage_table(a.dfa, g_smem, a.use_smem);
  const uint32_t match_lo = a.dfa.match_lo;
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < a.n_seg; t += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t s = exact[t];
    if (s == 0) continue;  // the run died further left
    const uint64_t lo = a.base + t * a.seg, hi = min(lo + a.seg, a.limit);  // a.limit: end of the window (<= n)
    uint64_t last = kNone;
    for (uint64_t q = lo; q < hi && s != 0; q++) {
      s = T.step(s, a.text[q]);
      if (s >= match_lo) last = q;
    }
    if (hi == a.limit && s != 0) {
      *alive_at_end = 1;  // the run goes on past the window (or meets the end of the text)
      if (a.limit == a.n && T.step_eof(s) >= match_lo) last = a.n;
    }
    if (last != kNone) atomicMax(best, (unsigned long long)last + 1);
  }
}

// result[0] = min first-match position, result[1..] = OR of masks.
__global__ void reduce_segments(const uint64_t* seg_first, const uint64_t* seg_mask, uint64_t n_seg, uint32_t mw,
                                unsigned long long* result) {
  uint64_t first = kNone;
  uint64_t acc[kMaxMaskWords] = {0, 0, 0, 0};
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < n_seg; t += (uint64_t)gridDim.x * blockDim.x) {
    first = min(first, seg_first[t]);
    if (seg_mask)
      for (uint32_t w = 0; w < mw; w++) acc[w] |= seg_mask[t * mw + w];
  }
  for (int o = 16; o; o >>= 1) {
    first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    for (uint32_t w = 0; w < kMaxMaskWords; w++) acc[w] |= __shfl_xor_sync(0xffffffffu, acc[w], o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (first != kNone) atomicMin(&result[0], (unsigned long long)first);
    for (uint32_t w = 0; w < mw; w++)
      if (acc[w]) atomicOr(&result[1 + w], (unsigned long long)acc[w]);
  }
}

// ---------------------------------------------------------------- walk_chunks --
// First match start in [pos, limit), or kNone.  Bit i of the bitmap stands for
// position i+1; position 0 is *flag0.
__device__ __forceinline__ uint64_t next_bit(const uint64_t* bm, const uint8_t* flag0, uint64_t pos, uint64_t limit) {
  if (pos >= limit) return kNone;
  if (pos == 0) {
    if (*flag0) return 0;
    pos = 1;
    if (pos >= limit) return kNone;
  }
  const uint64_t b_lo = pos - 1, b_hi = limit - 1;  // bits [b_lo, b_hi)
  uint64_t w = b_lo >> 6;
  const uint64_t last_w = (b_hi - 1) >> 6;
  uint64_t word = bm[w] & (~0ull << (b_lo & 63));
  for (;;) {
    if (word) {
      uint64_t b = (w << 6) + (uint64_t)(__ffsll((long long)word) - 1);
      return b < b_hi ? b + 1 : kNone;
    }
    if (w == last_w) return kNone;
    word = bm[++w];
  }
}

// End of the leftmost-first match anchored at s (src/dfa.rs:576-764 run on the
// anchored program): last position at which a match state was entered, with the
// one-byte delay and the EOF flush.  On an unanchored leftmost-first automaton: the
// end of the leftmost-first match found from s (the batched find_iter).
// halo_err: non-null when the buffer is a shard whose text continues past n (running
// into n then means the halo was too short, not end-of-text).
__device__ __forceinline__ uint64_t anchored_end(const DfaView& d, const Table& T, const uint8_t* text, uint64_t n, uint64_t s,
                                                 uint32_t* halo_err = nullptr, uint64_t cap = kNone) {
  uint32_t st = pick_start_fwd(d, text, n, s);
  uint64_t last = kNone;
  for (uint64_t q = s;; q++) {
    if (q - s > cap) return kTooLong;
    if (q >= n && halo_err) { *halo_err = 1; return last; }
    st = q < n ? T.step(st, __ldg(text + q)) : T.step_eof(st);
    if (st >= d.match_lo) last = q;
    if (st == 0 || q >= n) break;
  }
  return last;
}

// First position at which the automaton, started at s with the flags there, enters a match state (the
// shortest_match_at end, exec.rs:382-468); kNone when it dies first or reaches `bound`.
// halo_err: non-null when the text continues past n (a stream's window): a run that reaches n undecided sets it and
// returns kNone instead of taking the end-of-text step.
__device__ __forceinline__ uint64_t earliest_end(const DfaView& d, const Table& T, const uint8_t* text, uint64_t n, uint64_t s,
                                                 uint64_t bound = kNone, uint32_t* halo_err = nullptr) {
  uint32_t st = pick_start_fwd(d, text, n, s);
  for (uint64_t q = s; st != 0 && q < bound; q++) {
    if (q >= n && halo_err) { *halo_err = 1; return kNone; }
    st = q < n ? T.step(st, __ldg(text + q)) : T.step_eof(st);
    if (st >= d.match_lo) return q;
    if (q >= n) break;
  }
  return kNone;
}

// Start of the match ending at e, found the way the reference does it: the
// reverse DFA over the slice text[p..] (src/exec.rs:651-657), so position p is
// judged as beginning-of-text (SURVEY.md §8 hazard H1).
// floor: non-null when p is only a stand-in for a restart point left of a shard's buffer;
// set when the reverse scan reaches p alive, i.e. when the answer depends on what lies there.
__device__ __forceinline__ uint64_t slice_start(const DfaView& d, const uint8_t* text, uint64_t n, uint64_t p, uint64_t e,
                                                uint32_t* floor = nullptr) {
  const uint8_t* t = text + p;
  const uint64_t len = n - p;
  uint64_t at = e - p;
  uint32_t st = d.uniform_start ? d.start[32] : d.start[flags_reverse(t, len, at)];
  uint64_t last = kNone;
  if (st == 0) return kNone;
  while (at > 0) {
    at--;
    st = d.trans[st * d.stride + d.classes[t[at]]];
    if (st == 0) return last == kNone ? kNone : p + last;
    if (st >= d.match_lo) last = at + 1;
  }
  if (floor) *floor = 1;
  st = d.trans[st * d.stride + d.stride - 1];
  if (st >= d.match_lo) last = 0;
  return last == kNone ? kNone : p + last;
}

__device__ __forceinline__ uint64_t next_utf8(const uint8_t* text, uint64_t n, uint64_t i) {  // src/utf8.rs:24-40
  if (i >= n) return i + 1;
  uint32_t b = text[i];
  return i + (b <= 0x7F ? 1 : b <= 0xDF ? 2 : b <= 0xEF ? 3 : 4);
}

// Generic anchored runner: class-indexed table (shared memory when it fits), any start flags.
struct GenericRunner {
  Table T;
  __device__ __forceinline__ uint64_t end_from(const WalkArgs& a, uint64_t s, uint64_t cap = kNone) const {
    return anchored_end(a.fwd, T, a.text, a.n, s, a.text_continues ? a.err_flag : nullptr, cap);
  }
};
// Fast anchored runner: byte-indexed XOR-swizzled table in shared memory (one LDS per
// byte, see scan_rev_fast), uniform start state, text taken 16 bytes at a time from
// three aligned 8-byte loads so a typical match costs one memory round trip.
// The anchored run on the full class-indexed table in global memory: where a FastRunner
// lane goes when the haystack leaves the hot set (e.g. a non-ASCII byte under \w).
// (scalar arguments only: a reference to the kernel's parameter block would make every
// thread copy it to its stack.)  FastRunner patterns have a uniform start state.
__device__ __noinline__ uint64_t slow_anchored_end(const uint16_t* trans, const uint8_t* classes, uint32_t stride, uint32_t match_lo,
                                                   uint32_t start, const uint8_t* text, uint64_t n, uint64_t s, uint32_t* halo_err, uint64_t cap) {
  uint32_t st = start;
  uint64_t last = kNone;
  for (uint64_t q = s;; q++) {
    if (q - s > cap) return kTooLong;
    if (q >= n && halo_err) { *halo_err = 1; return last; }
    st = q < n ? trans[st * stride + classes[__ldg(text + q)]] : trans[st * stride + stride - 1];
    if (st >= match_lo) last = q;
    if (st == 0 || q >= n) break;
  }
  return last;
}
struct FastRunner {
  uint32_t tb, thr, start_e;  // table address, first match row, start row
  const uint16_t* eof;  // by hot id, value in full numbering
  uint32_t match_lo;    // full numbering (for the EOF successor)
  static __device__ __forceinline__ uint64_t slow(const WalkArgs& a, uint64_t s, uint64_t cap) {
    return slow_anchored_end(a.fwd.trans, a.fwd.classes, a.fwd.stride, a.fwd.match_lo, a.fwd.start[32], a.text, a.n, s,
                             a.text_continues ? a.err_flag : nullptr, cap);
  }
  __device__ __forceinline__ uint64_t end_from(const WalkArgs& a, uint64_t s, uint64_t cap = kNone) const {
    uint32_t e = start_e;
    uint64_t last = kNone;
    const uint32_t live = 2;  // rows 0 (dead) and 1 (trap) end the run
    for (uint64_t q = s;; q += 16) {
      if (q - s > cap) return kTooLong;
      const uint64_t al = q & ~7ull;
      const uint64_t* wp = reinterpret_cast<const uint64_t*>(a.text + al);
      const uint32_t sh = (uint32_t)(q & 7) * 8;
      if (al + 24 <= a.n) {
        // common case: the whole 16-byte window lies inside the haystack -- 32-bit
        // bookkeeping only (offset of the last match state inside the window)
        const uint64_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
        const uint32_t x0 = __funnelshift_r((uint32_t)w0, (uint32_t)(w0 >> 32), sh);
        const uint32_t x1 = __funnelshift_r((uint32_t)(w0 >> 32), (uint32_t)w1, sh);
        const uint32_t x2 = __funnelshift_r((uint32_t)w1, (uint32_t)(w1 >> 32), sh);
        const uint32_t x3 = __funnelshift_r((uint32_t)(w1 >> 32), (uint32_t)w2, sh);
        const uint32_t x4 = __funnelshift_r((uint32_t)w2, (uint32_t)(w2 >> 32), sh);
        // sh in {0,8,..,56}: for sh >= 32 the window starts one word later
        const bool up = sh >= 32;
        const uint32_t v[4] = {up ? x1 : x0, up ? x2 : x1, up ? x3 : x2, up ? x4 : x3};
        uint32_t lj = ~0u;
        bool died = false;
#pragma unroll
        for (int g = 0; g < 4; g++) {
          e = hot_next<0>(tb, v[g], e); if (e >= thr) lj = 4 * g + 0;
          e = hot_next<1>(tb, v[g], e); if (e >= thr) lj = 4 * g + 1;
          e = hot_next<2>(tb, v[g], e); if (e >= thr) lj = 4 * g + 2;
          e = hot_next<3>(tb, v[g], e); if (e >= thr) lj = 4 * g + 3;
          if (e < live) { died = true; break; }
        }
        if (e == 1) return slow(a, s, cap);  // trap: left the hot set
        if (lj != ~0u) last = q + lj;
        if (died) return last;
        continue;
      }
      const uint64_t w0 = al < a.n ? __ldg(wp) : 0, w1 = al + 8 < a.n ? __ldg(wp + 1) : 0, w2 = al + 16 < a.n ? __ldg(wp + 2) : 0;
      const uint64_t lo = sh ? (w0 >> sh) | (w1 << (64 - sh)) : w0;
      const uint64_t hi = sh ? (w1 >> sh) | (w2 << (64 - sh)) : w1;
      const uint64_t avail = a.n - q;  // bytes before EOF (q <= n)
#pragma unroll 1
      for (int j = 0; j < 16; j++) {
        if ((uint64_t)j >= avail) {  // EOF step (dfa.rs:748-763)
          if (a.text_continues) { *a.err_flag = 1; return last; }
          if (eof[e] >= match_lo) last = a.n;
          return last;
        }
        const uint32_t byte = (uint32_t)((j < 8 ? lo >> (8 * j) : hi >> (8 * (j - 8))) & 0xFF);
        e = hot_next_b(tb, byte, e);
        if (e >= thr) last = q + j;
        if (e < live) return e == 1 ? slow(a, s, cap) : last;
      }
    }
  }
};

// Fixed-length patterns (min == max match length, e.g. the regex-dna variants or
// `Holmes|Watson`): a candidate start s is known to begin a match, and every match has
// the same length, so the leftmost-first end is s + L without touching the haystack.
struct FixedLenRunner {
  uint64_t len;
  __device__ __forceinline__ uint64_t end_from(const WalkArgs&, uint64_t s, uint64_t = kNone) const { return s + len; }
};

// Chain state of the find_iter iterator (re_trait.rs:174-179).
struct Chain {
  uint64_t p, lm;  // next search position, end of the previous match (kNone = none)
  bool chain;      // p is a real restart point of the reference iterator
};

// End of the match anchored at s for a chunk walk.  Speculative walks give up early (kSpecRunCap);
// walks from an exact entry state take matches of up to exact_cap bytes themselves, look longer
// ones up in the table of runs the host has measured with a parallel scan, and otherwise ask for
// that (long_req) -- in both cases kTooLong defers the chunk.
// trip_cap: inside a voting trip loop (see kTripRunCap); kPending then means "longer than that, ask again".
template <typename Runner>
__device__ __forceinline__ uint64_t run_end(const WalkArgs& a, const Runner& T, uint64_t s, bool exact, uint64_t trip_cap = kNone) {
  if (exact)
    for (uint32_t i = 0; i < a.n_long; i++)
      if (a.long_tab[2 * i] == s) return a.long_tab[2 * i + 1];
  const uint64_t cap = exact ? a.exact_cap : kSpecRunCap;
  const uint64_t e = T.end_from(a, s, min(cap, trip_cap));
  if (e == kTooLong && trip_cap < cap) return kPending;
  if (e == kTooLong && exact) atomicMin(a.long_req, (unsigned long long)s);
  return e;
}

template <typename Runner>
__device__ __forceinline__ uint64_t chunk_walk_simple(const WalkArgs& a, const Runner& T, uint64_t k, Chain& c, uint64_t* first_cand,
                                                      uint64_t* dst, uint64_t w_at, uint64_t limit, uint64_t nz, uint32_t lanes);
__device__ __forceinline__ uint64_t chunk_walk_lean(const WalkArgs& a, const FastRunner& T, uint64_t k, Chain& c, uint64_t* first_cand,
                                                    uint64_t* dst, uint64_t w_at, uint64_t limit, uint64_t nz, uint32_t lanes);

// The chain over one chunk (bits [cb, ce) <-> positions [cb+1, ce], plus position 0
// for the chunk that starts the haystack).  One flat loop -- find the next candidate,
// run the anchored automaton, advance the iterator -- so that the lanes of a warp
// stay in the same phase (the nested per-word version ran at 5.7 of 32 lanes active).
// Spans are written to dst[w_at + i] while w_at + i < limit.  Returns the match count.
// nz: bit j set iff bitmap word j of the chunk may be non-zero (all ones when unknown);
// lets the fused scan kernel skip the words it already knows to be empty.
// lanes: the lanes of the warp that call this together (0 = unknown): the simple walk then votes
// once per trip, which keeps them converged -- left to itself the compiler lets lanes drift apart
// after the divergent exits of a run and the trip loop executes twice per match.
template <typename Runner>
__device__ __forceinline__ uint64_t chunk_walk(const WalkArgs& a, const Runner& T, uint64_t k, Chain& c, uint64_t* first_cand,
                                               uint64_t* dst, uint64_t w_at, uint64_t limit, uint64_t nz = ~0ull, uint32_t lanes = 0) {
  if (!a.emulate_slice && !a.can_match_empty && a.chunk <= 4096) {
    if constexpr (std::is_same<Runner, FastRunner>::value) {
      bool aligned = (((uintptr_t)a.text | (uintptr_t)dst) & 31) == 0 && !(w_at & 1);
      if (lanes) aligned = __all_sync(lanes, aligned);  // the lanes that vote together take the same version
      if (aligned) return chunk_walk_lean(a, T, k, c, first_cand, dst, w_at, limit, nz, lanes);
    }
    return chunk_walk_simple(a, T, k, c, first_cand, dst, w_at, limit, nz, lanes);
  }
  const uint64_t cb = a.base + k * (uint64_t)a.chunk;
  const uint64_t ce = min(cb + a.chunk, a.limit);
  uint64_t total = 0;
  uint64_t fc = kNone;
  const bool exact = c.chain;  // only an exact entry state justifies a long run
  uint64_t cached_w = kNone, word = 0;
  uint64_t pf_w = kNone, pf_word = 0;  // next candidate word, load issued ahead of use
  const uint64_t w0 = cb >> 6, w_end = (ce + 63) >> 6;
  // first word at or after `wi` that may be non-zero (w_end if none)
  auto next_word = [&](uint64_t wi) -> uint64_t {
    if (wi >= w_end) return w_end;
    const uint64_t rel = wi - w0;
    if (rel >= 64) return wi;
    const uint64_t ahead = nz >> rel;
    if (ahead == 0) return rel + 64 >= w_end - w0 ? w_end : w0 + 64;
    return wi + (uint64_t)(__ffsll((long long)ahead) - 1);
  };
  bool at_zero = c.p == 0 && cb == 0 && *a.flag0;  // position 0 has no bitmap bit
  uint64_t q = 0;  // candidates below q were no match start (candidate-start bitmaps are a superset)
  while (c.p != kNone) {
    uint64_t s;
    if (at_zero) {
      s = 0;
      at_zero = false;
    } else {
      // next candidate position >= max(p, q, cb + 1): bit index = position - 1
      uint64_t bit = max(max(c.p, q), cb + 1) - 1;
      uint64_t m = 0;
      while (bit < ce) {
        uint64_t wi = bit >> 6;
        const uint64_t nw = next_word(wi);
        if (nw != wi) { wi = nw; bit = wi << 6; if (bit >= ce) break; }
        if (wi != cached_w) {
          word = wi == pf_w ? pf_word : a.bitmap[wi];
          cached_w = wi;
          pf_w = next_word(wi + 1);  // start fetching the following candidate word now
          if (pf_w < w_end) pf_word = a.bitmap[pf_w];
        }
        m = word & (~0ull << (bit & 63));
        if (m) break;
        bit = (wi + 1) << 6;
      }
      if (bit >= ce) break;
      s = (bit & ~63ull) + (uint64_t)__ffsll((long long)m);
    }
    if (fc == kNone) fc = s;
    const uint64_t e = run_end(a, T, s, exact);
    if (e == kTooLong) { *first_cand = kTooLong; return 0; }  // deferred: see kSpecRunCap
    if (e == kNone) {  // no match starts at s (a candidate start): the iterator state stays, the walk moves on
      if (fc == s) fc = kNone;
      q = s + 1;
      continue;
    }
    uint64_t ms = s;
    if (a.emulate_slice && c.chain && e != c.p) {
      // exec.rs:647-657: an empty match at the restart point short-circuits; otherwise
      // the start comes from the reverse DFA over text[p..].
      ms = slice_start(a.rev, a.text, a.n, c.p, e, c.p == a.clamp_p ? a.floor_flag : nullptr);
      if (ms == kNone) { c.p = kNone; break; }  // NoMatch => find_at None => the iteration stops
    }
    c.chain = true;
    if (ms == e) {
      c.p = a.utf8 ? next_utf8(a.text, a.n, e) : e + 1;
      if (e == c.lm) continue;  // re_trait.rs:210-214
    } else {
      c.p = e;
    }
    c.lm = e;
    if (w_at + total < limit) { dst[2 * (w_at + total)] = ms; dst[2 * (w_at + total) + 1] = e; }
    total++;
  }
  *first_cand = fc;
  return total;
}

// chunk_walk for the common pattern class -- no empty matches, no slice emulation --
// where every candidate yields a span and the iterator simply continues at the match
// end.  Same contract as chunk_walk; bit positions are kept relative to the chunk in
// 32 bits and the chunk's non-zero words are visited through the `nz` mask, which
// roughly halves the instructions per match.  Requires chunks of at most 64 words.
template <typename Runner>
__device__ __forceinline__ uint64_t chunk_walk_simple(const WalkArgs& a, const Runner& T, uint64_t k, Chain& c, uint64_t* first_cand,
                                                      uint64_t* dst, uint64_t w_at, uint64_t limit, uint64_t nz, uint32_t lanes) {
  const uint64_t cb = a.base + k * (uint64_t)a.chunk;
  const uint64_t ce = min(cb + a.chunk, a.limit);
  const uint32_t nbits = (uint32_t)(ce - cb);
  const uint64_t* bm = a.bitmap + (cb >> 6);  // cb is a multiple of 64
  uint64_t* o = dst + 2 * w_at;
  uint32_t room = limit > w_at ? (uint32_t)min(limit - w_at, (uint64_t)0xFFFFFFFFu) : 0u;
  uint32_t total = 0;
  uint64_t fc = kNone;
  const bool exact = c.chain;
  // Spans leave two at a time as whole 32-byte sectors when the destination allows it
  // (staging areas do): the even span of a pair waits in registers for the odd one.
  const bool pair_stores = ((uintptr_t)o & 31) == 0;
  uint64_t held_s = 0, held_e = 0;
  auto emit = [&](uint64_t ms, uint64_t e) {
    if (pair_stores) {
      if (!(total & 1u)) { held_s = ms; held_e = e; }
      else if (total < room) st_sector(o + 2 * (uint64_t)(total - 1), held_s, held_e, ms, e);
      else if (total - 1 < room) *reinterpret_cast<ulonglong2*>(o + 2 * (uint64_t)(total - 1)) = make_ulonglong2(held_s, held_e);
    } else if (total < room) {
      if (((uintptr_t)o & 15) == 0) {
        *reinterpret_cast<ulonglong2*>(o + 2 * (uint64_t)total) = make_ulonglong2(ms, e);
      } else {
        o[2 * (uint64_t)total] = ms;
        o[2 * (uint64_t)total + 1] = e;
      }
    }
    total++;
  };
  auto flush = [&]() {  // the unpaired last span
    if (pair_stores && (total & 1u) && total - 1 < room)
      *reinterpret_cast<ulonglong2*>(o + 2 * (uint64_t)(total - 1)) = make_ulonglong2(held_s, held_e);
  };
  bool too_long = false;
  if (c.p == kNone) { *first_cand = fc; return 0; }  // (never among `lanes`)
  if (c.p == 0 && cb == 0 && *a.flag0) {  // position 0 has no bitmap bit
    fc = 0;
    const uint64_t e = run_end(a, T, 0, exact);
    if (e == kTooLong) too_long = true;
    else if (e == kNone) fc = kNone;  // a candidate that is no match start: as if its bit were clear
    else { emit(0, e); c.p = c.lm = e; c.chain = true; }
  }
  // bit r of the chunk <-> position cb + r + 1
  uint32_t r = c.p > cb + 1 ? (uint32_t)min(c.p - cb - 1, (uint64_t)nbits) : 0u;
  if (nbits < 64 * 64) nz &= (1ull << ((nbits + 63) >> 6)) - 1;
  uint64_t rem = r < nbits ? nz & (~0ull << (r >> 6)) : 0;  // words still to visit
  uint32_t cw = 0;
  uint64_t cur = 0;
  bool pending = false;
  auto trip = [&]() -> bool {  // one candidate; false when the chunk is through
    if (cur == 0) {
      if (rem == 0) return false;
      cw = (uint32_t)__ffsll((long long)rem) - 1;
      rem &= rem - 1;
      cur = bm[cw];
      if (cw == (r >> 6)) cur &= ~0ull << (r & 63);
      if (cur == 0) return true;  // rare; otherwise fall through: one trip per match keeps the lanes of a warp in phase
    }
    const uint32_t sr = cw * 64 + (uint32_t)__ffsll((long long)cur) - 1;
    const uint64_t s = cb + sr + 1;
    if (fc == kNone) fc = s;
    const uint64_t e = pending ? run_end(a, T, s, exact) : run_end(a, T, s, exact, lanes ? kTripRunCap : kNone);
    pending = e == kPending;
    if (pending) return false;  // the same candidate again, without the trip cap, once the warp is through its short runs
    if (e == kTooLong) { too_long = true; return false; }
    if (e == kNone) {  // a candidate that is no match start: as if its bit were clear
      cur &= cur - 1;
      if (fc == s) fc = kNone;
      return true;
    }
    emit(s, e);
    c.p = c.lm = e;
    c.chain = true;
    const uint64_t er = e - 1 - cb;  // next candidate bit >= er
    if (er >= nbits) return false;
    r = (uint32_t)er;
    const uint32_t ew = r >> 6;
    if (ew == cw) {
      cur &= ~0ull << (r & 63);
    } else {
      cur = 0;
      rem &= ~0ull << ew;
    }
    return true;
  };
  if (lanes) {
    bool active = !too_long;
    for (;;) {
      while (__any_sync(lanes, active))
        if (active) active = trip();
      if (!__any_sync(lanes, pending)) break;
      if (pending) active = trip();  // the long runs of the warp, side by side
    }
  } else if (!too_long) {
    while (trip()) {}
  }
  if (too_long) { *first_cand = kTooLong; return 0; }
  flush();
  *first_cand = fc;
  return total;
}

// chunk_walk_simple once more for the fast table runner, the walk the headline kernel spends a third
// of its time in: positions relative to the chunk in 32 bits, the first 16 bytes of every anchored
// run without a branch (rows 0 -- dead -- and 1 -- trap -- are absorbing, so running past the end of
// a match is harmless), everything unusual (a run still alive after 16 bytes, the trap row, the
// last bytes of the haystack, long-run caps) handed to run_end.  About half the instructions per
// match of the general version; same contract, dst must be the 32-byte aligned staging area.
__device__ __forceinline__ uint64_t chunk_walk_lean(const WalkArgs& a, const FastRunner& T, uint64_t k, Chain& c, uint64_t* first_cand,
                                                    uint64_t* dst, uint64_t w_at, uint64_t limit, uint64_t nz, uint32_t lanes) {
  const uint64_t cb = a.base + k * (uint64_t)a.chunk;
  const uint64_t ce = min(cb + a.chunk, a.limit);
  const uint32_t nbits = (uint32_t)(ce - cb);
  const uint64_t* bm = a.bitmap + (cb >> 6);
  const uint8_t* tb8 = a.text + cb;  // cb is a multiple of 64 and the haystack is 16-byte aligned
  // a 32-byte window read at relative offset x (multiple of 16) is inside the haystack iff x < safe
  const uint64_t left = a.n - cb;
  const uint32_t safe = left >= 32 ? (uint32_t)min(left - 31, (uint64_t)0x7FFFFFFFu) : 0u;
  ulonglong2* o = reinterpret_cast<ulonglong2*>(dst) + w_at;
  const uint32_t room = limit > w_at ? (uint32_t)min(limit - w_at, (uint64_t)0xFFFFFFFFu) : 0u;
  const bool exact = c.chain;
  uint32_t total = 0, fc_rel = ~0u;
  uint64_t held_s = 0, held_e = 0, last_e = kNone;
  bool too_long = false;
  auto emit = [&](uint64_t ms, uint64_t e) {  // spans leave two at a time as whole 32-byte sectors
    if (!(total & 1u)) { held_s = ms; held_e = e; }
    else if (total < room) st_sector(reinterpret_cast<uint64_t*>(o + (total - 1)), held_s, held_e, ms, e);
    else if (total - 1 < room) o[total - 1] = make_ulonglong2(held_s, held_e);
    total++;
  };
  uint64_t fc0 = kNone;
  if (c.p == 0 && cb == 0 && *a.flag0) {  // position 0 has no bitmap bit
    fc0 = 0;
    const uint64_t e = run_end(a, T, 0, exact);
    if (e == kTooLong) too_long = true;
    else if (e == kNone) fc0 = kNone;  // a candidate that is no match start: as if its bit were clear
    else { emit(0, e); c.p = last_e = e; c.chain = true; }
  }
  uint32_t r = c.p > cb + 1 ? (uint32_t)min(c.p - cb - 1, (uint64_t)nbits) : 0u;
  if (nbits < 64 * 64) nz &= (1ull << ((nbits + 63) >> 6)) - 1;
  uint64_t rem = r < nbits ? nz & (~0ull << (r >> 6)) : 0;
  // Candidate words come one ahead: while the candidates of word cw are walked, the chunk's next
  // non-zero word nw is already on its way (nxt), and the haystack line of the likely next
  // candidate -- the first bit after the current run of ones -- is prefetched into L1.  Without
  // this every trip paid two L2 round trips in a row (bitmap word, then haystack bytes).
  uint32_t cw = 0, nw = 64;  // nw == 64: nothing preloaded; bit nw of rem is already taken
  uint64_t cur = 0, nxt = 0;
  auto preload = [&]() {
    if (rem) { nw = (uint32_t)__ffsll((long long)rem) - 1; rem &= rem - 1; nxt = bm[nw]; }
    else nw = 64;
  };
  const uint32_t tb = T.tb, thr = T.thr, start_e = T.start_e;
  bool pending = false;
  auto trip = [&]() -> bool {
    if (cur == 0) {
      if (nw == 64) preload();
      if (nw == 64) return false;
      cw = nw;
      cur = nxt;
      preload();
      if (cw == (r >> 6)) cur &= ~0ull << (r & 63);
      if (cur == 0) return true;
    }
    const uint32_t s_rel = cw * 64 + (uint32_t)__ffsll((long long)cur);  // bit index + 1
    if (fc_rel == ~0u) fc_rel = s_rel;
    {
      const uint64_t after_run = cur & (cur + (cur & (0 - cur)));  // the candidates of this word behind the current run of ones
      const uint32_t g = after_run ? cw * 64 + (uint32_t)__ffsll((long long)after_run)
                                   : (nw != 64 && nxt) ? nw * 64 + (uint32_t)__ffsll((long long)nxt) : 0u;
      if (g != 0 && g < left) asm volatile("prefetch.global.L1 [%0];" ::"l"(tb8 + g));
    }
    const uint32_t al = s_rel & ~15u;
    uint64_t e_abs;
    bool fast_done = false;
    if (al < safe) {
      // two aligned 16-byte loads (two L1 wavefronts per lane; three 8-byte loads were three), then the 16
      // bytes from s on: word offset through two rounds of selects, byte offset through funnel shifts
      const uint4 p0 = ldg128(tb8 + al), p1 = ldg128(tb8 + al + 16);
      const bool by2 = (s_rel & 8u) != 0, by1 = (s_rel & 4u) != 0;
      const uint32_t sh = (s_rel & 3u) * 8u;
      const uint32_t a0 = by2 ? p0.z : p0.x, a1 = by2 ? p0.w : p0.y, a2 = by2 ? p1.x : p0.z, a3 = by2 ? p1.y : p0.w,
                     a4 = by2 ? p1.z : p1.x, a5 = by2 ? p1.w : p1.y;
      const uint32_t b0 = by1 ? a1 : a0, b1 = by1 ? a2 : a1, b2 = by1 ? a3 : a2, b3 = by1 ? a4 : a3, b4 = by1 ? a5 : a4;
      const uint32_t v0 = __funnelshift_r(b0, b1, sh), v1 = __funnelshift_r(b1, b2, sh);
      uint32_t e = start_e, lj = ~0u;
#define RB_LEAN_WORD(V, J0)                                         \
      e = hot_next<0>(tb, V, e); if (e >= thr) lj = J0 + 0;         \
      e = hot_next<1>(tb, V, e); if (e >= thr) lj = J0 + 1;         \
      e = hot_next<2>(tb, V, e); if (e >= thr) lj = J0 + 2;         \
      e = hot_next<3>(tb, V, e); if (e >= thr) lj = J0 + 3;
      RB_LEAN_WORD(v0, 0) RB_LEAN_WORD(v1, 4)
      if (e >= 2) {  // still alive after 8 bytes: the second half of the window
        const uint32_t v2 = __funnelshift_r(b2, b3, sh), v3 = __funnelshift_r(b3, b4, sh);
        RB_LEAN_WORD(v2, 8) RB_LEAN_WORD(v3, 12)
      }
#undef RB_LEAN_WORD
      if (e == 0 && lj != ~0u) { e_abs = cb + s_rel + lj; fast_done = true; }
    }
    if (!fast_done) {  // rare: longer than 16 bytes, left the hot set, near the end of the haystack
      e_abs = pending ? run_end(a, T, cb + s_rel, exact) : run_end(a, T, cb + s_rel, exact, lanes ? kTripRunCap : kNone);
      pending = e_abs == kPending;
      if (pending) return false;  // the same candidate again, without the trip cap, once the warp is through its short runs
      if (e_abs == kTooLong) { too_long = true; return false; }
      if (e_abs == kNone) {  // a candidate that is no match start: as if its bit were clear
        cur &= cur - 1;
        if (fc_rel == s_rel) fc_rel = ~0u;
        return true;
      }
    }
    emit(cb + s_rel, e_abs);
    last_e = e_abs;
    const uint64_t er = e_abs - 1 - cb;  // next candidate bit >= er
    if (er >= nbits) return false;
    r = (uint32_t)er;
    const uint32_t ew = r >> 6;
    if (ew == cw) {
      cur &= ~0ull << (r & 63);
    } else {
      cur = 0;
      rem &= ~0ull << ew;
      if (nw < ew) nw = 64;  // (64 is never below ew)
    }
    return true;
  };
  if (lanes) {
    bool active = !too_long;
    for (;;) {
      while (__any_sync(lanes, active))
        if (active) active = trip();
      if (!__any_sync(lanes, pending)) break;
      if (pending) active = trip();  // the long runs of the warp, side by side
    }
  } else if (!too_long) {
    while (trip()) {}
  }
  if (too_long) { *first_cand = kTooLong; return 0; }
  if ((total & 1u) && total - 1 < room) o[total - 1] = make_ulonglong2(held_s, held_e);
  if (last_e != kNone) { c.p = c.lm = last_e; c.chain = true; }
  *first_cand = fc0 != kNone ? fc0 : fc_rel != ~0u ? cb + fc_rel : kNone;
  return total;
}

// Runner set-up shared by the walk kernels: 0 = generic, 1 = fast table, 2 = fixed length.
template <int FAST>
struct RunnerSetup;
template <>
struct RunnerSetup<2> {
  using type = FixedLenRunner;
  static __device__ __forceinline__ type make(const WalkArgs& a) {
    FixedLenRunner r;
    r.len = a.fixed_len;
    return r;
  }
};
template <>
struct RunnerSetup<0> {
  using type = GenericRunner;
  static __device__ __forceinline__ type make(const WalkArgs& a) {
    GenericRunner r;
    r.T = stage_table(a.fwd, g_smem, a.use_smem);
    return r;
  }
};
template <>
struct RunnerSetup<1> {
  using type = FastRunner;
  static __device__ __forceinline__ type make(const WalkArgs& a) {
    FastRunner r;
    r.tb = ((uint32_t)__cvta_generic_to_shared(g_smem) + 255u) & ~255u;
    hot_stage(a.fwd_hot, r.tb);
    __syncthreads();
    r.thr = a.fwd_hot.match_lo;
    r.start_e = a.fwd_hot.start;
    r.eof = a.fwd_hot.eof;
    r.match_lo = a.fwd.match_lo;
    return r;
  }
};

// What every walk leaves behind for the stitch: exit state, counts, and whether the chunk
// holds any candidate at all (a speculative walk that met none is IDENT: the iterator
// passes through it unchanged whatever its entry state).
__device__ __forceinline__ void finish_chunk(const WalkArgs& a, uint64_t k, const Chain& c, uint64_t total, uint64_t fc, bool spec) {
  a.out_p[k] = c.p;
  a.out_lm[k] = c.lm;
  a.skip[k] = 0;
  if (fc == kTooLong) {  // the walk gave up on a long match (kSpecRunCap): nothing staged, the stitch decides
    a.count[k] = 0;
    a.first_cand[k] = kNone;
    a.meta[k] = kChunkDeferred << 30;
    return;
  }
  a.count[k] = total;
  a.first_cand[k] = fc;
  a.meta[k] = (uint32_t)min(total, (uint64_t)kMetaCount) | ((spec && fc == kNone ? kChunkIdent : kChunkOk) << 30);
}

// One thread per chunk: walk the chain speculatively (or from a given entry state),
// staging up to stage_cap spans per chunk.  With a dirty list (after stitch_check)
// only the listed chunks are walked again, densely packed into warps.
template <int FAST>
__global__ void __launch_bounds__(256) walk_chunks(WalkArgs a) {
  const auto R = RunnerSetup<FAST>::make(a);
  const uint64_t work = a.dirty_list ? (uint64_t)*a.n_dirty : a.n_chunks;
  for (uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; idx < work;
       idx += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t k = a.dirty_list ? a.dirty_list[idx] : idx;
    Chain c;
    c.p = a.in_p[k];
    c.lm = a.in_lm[k];
    c.chain = c.p != kSpec;
    const bool spec = !c.chain;
    if (spec) { c.p = a.base + k * (uint64_t)a.chunk + 1; c.lm = kNone; }
    uint64_t fc = kNone, total = 0;
    const uint32_t walkers = __ballot_sync(__activemask(), c.p != kNone);
    if (c.p != kNone) total = chunk_walk(a, R, k, c, &fc, a.stage, k * (uint64_t)a.stage_cap, (k + 1) * (uint64_t)a.stage_cap, ~0ull, walkers);
    finish_chunk(a, k, c, total, fc, spec);
  }
}
template __global__ void walk_chunks<0>(WalkArgs);
template __global__ void walk_chunks<1>(WalkArgs);
template __global__ void walk_chunks<2>(WalkArgs);

// Staged spans -> final array at the prefix-summed offsets.  A warp takes 32 consecutive
// chunks and copies them one after the other with all lanes (coalesced 16-byte spans);
// a chunk that overflowed its staging slots is walked again by one lane, writing straight
// to the output.
template <int FAST>
__global__ void __launch_bounds__(256) compact_spans(WalkArgs a) {
  const auto R = RunnerSetup<FAST>::make(a);
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp0 = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  const ulonglong2* stage = reinterpret_cast<const ulonglong2*>(a.stage);
  ulonglong2* dst = reinterpret_cast<ulonglong2*>(a.out);
  for (uint64_t g = warp0; g * 32 < a.n_chunks; g += n_warps) {
    const uint64_t k = g * 32 + lane;
    const uint64_t my_cnt = k < a.n_chunks ? a.count[k] : 0;
    const uint64_t my_at = k < a.n_chunks ? a.offset[k] : 0;
    const uint32_t my_skip = k < a.n_chunks ? a.skip[k] : 0;
    const uint32_t walkers = __ballot_sync(0xffffffffu, my_cnt > a.stage_cap);
    if (my_cnt > a.stage_cap) {  // rare: dense chunk, redo it in place (such a chunk is never trimmed: count == walk count)
      Chain c;
      c.p = a.in_p[k];
      c.lm = a.in_lm[k];
      c.chain = c.p != kSpec;
      if (!c.chain) { c.p = a.base + k * (uint64_t)a.chunk + 1; c.lm = kNone; }
      uint64_t fc;
      chunk_walk(a, R, k, c, &fc, a.out, my_at, a.cap, ~0ull, walkers);  // voting together: without it the lanes drift apart, 13x slower on `\w+`
    }
    __syncwarp();
    // The staged spans of the warp's 32 chunks as ONE list: lane i of a row takes element 32 * row + i whatever
    // chunk it belongs to (a chunk holds ~19 spans on the headline pattern: one chunk per instruction left a
    // third of the lanes idle and the stores in pieces).  Four rows per trip keep four loads per lane in flight.
    const uint32_t copy_cnt = my_cnt <= a.stage_cap ? (uint32_t)my_cnt : 0u;  // overflowed chunks were written above
    uint32_t pre = copy_cnt;  // exclusive prefix over the lanes
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, pre, o);
      if ((int)lane >= o) pre += y;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, pre, 31);
    pre -= copy_cnt;
    for (uint32_t row0 = 0; row0 < total; row0 += 128) {
      ulonglong2 v[4];
      uint64_t to[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const uint32_t i = row0 + 32 * u + lane;
        // the chunk of element i: the last lane whose prefix is <= i (chunks without spans share a prefix with
        // their successor and are passed over)
        uint32_t j = 0;
#pragma unroll
        for (int step = 16; step; step >>= 1) {
          const uint32_t cand = j + step;
          const uint32_t pv = __shfl_sync(0xffffffffu, pre, cand & 31);
          if (cand < 32 && pv <= i) j = cand;
        }
        const uint32_t pj = __shfl_sync(0xffffffffu, pre, j);
        const uint32_t sj = __shfl_sync(0xffffffffu, my_skip, j);
        const uint64_t aj = __shfl_sync(0xffffffffu, my_at, j);
        to[u] = ~0ull;
        if (i < total) {
          v[u] = stage[(g * 32 + j) * (uint64_t)a.stage_cap + sj + (i - pj)];
          to[u] = aj + (i - pj);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (to[u] < a.cap) dst[to[u]] = v[u];
    }
  }
}
template __global__ void compact_spans<0>(WalkArgs);
template __global__ void compact_spans<1>(WalkArgs);
template __global__ void compact_spans<2>(WalkArgs);

// ---------------------------------------------------------- literal prefilter --
// The GPU analogue of the reference's literal searchers (src/literals.rs:92-102 LiteralSearcher,
// :353-371 memchr sets, :466-489 FreqyPacked; Teddy src/simd_accel/teddy128.rs:435-675) and of the
// prefix skip of the DFA loop (src/dfa.rs:700-711): for patterns that cannot match without one of
// a few RARE bytes at a fixed offset (`Holmes|Watson`, `Sherlock|Holmes`, `Sher[a-z]+|Hol[a-z]+`),
// the haystack is streamed once with coalesced 16-byte loads and tested for those bytes with
// word-wide arithmetic -- no table look-up and no loop-carried dependency, so the loads of a
// warp are always in flight -- and only the hits are looked at again:
//   1. the byte is confirmed, and the bytes at the first offsets of the would-be match are
//      tested against the sets the automaton allows there (the Teddy fingerprint idea);
//   2. survivors run the anchored leftmost-first automaton (exec_at) from the candidate start:
//      that decides whether a match starts there and where it ends, so results are the DFA's;
//   3. the warp applies the find_iter rule (re_trait.rs:197-220) to its chunk's matches in
//      position order, speculatively entered like every other chunk walk; stitch, prefix sums
//      and compaction are the common ones.
// One warp per chunk of a.chunk bytes; chunk k owns the candidates whose scanned byte lies in
// [base + k*chunk, base + (k+1)*chunk), i.e. the match starts `o` bytes before.
__device__ __forceinline__ uint4 ldg128_stream(const uint8_t* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
// flag (bit 7 of each byte) where a byte of w equals the byte replicated in cc; flags above a
// true hit may be spurious, the lowest one never is -- hits are confirmed anyway
__device__ __forceinline__ uint32_t swar_eq(uint32_t w, uint32_t cc) {
  const uint32_t x = w ^ cc;
  return (x - 0x01010101u) & ~x & 0x80808080u;
}
template <int NB>
__device__ __forceinline__ uint32_t swar_any(const uint32_t (&cc)[4], uint32_t w) {
  uint32_t t = swar_eq(w, cc[0]);
  if (NB > 1) t |= swar_eq(w, cc[1]);
  if (NB > 2) t |= swar_eq(w, cc[2]);
  if (NB > 3) t |= swar_eq(w, cc[3]);
  return t;
}
__device__ __forceinline__ uint32_t flags_to_bits(uint32_t t) {  // bits 7,15,23,31 -> bits 0..3
  return (((t >> 7) & 0x01010101u) * 0x01020408u) >> 24;
}

// The verifier, out of line: one copy of the automaton loop however many call sites, and the
// streaming loop stays small (the first version inlined it three times and starved on
// instruction fetch: ncu "no instruction" 7.9 stalls per issue).
template <typename Runner>
__device__ __noinline__ uint64_t pf_verify(const WalkArgs* a, const Runner* R, uint64_t s, bool exact) {
  if (exact)
    for (uint32_t i = 0; i < a->n_long; i++)
      if (a->long_tab[2 * i] == s) return a->long_tab[2 * i + 1];
  return R->end_from(*a, s, exact ? a->exact_cap : kSpecRunCap);  // kTooLong: the caller defers the chunk (run_end)
}

// Is a match possible with its scanned byte at q?  Tests the bytes at the first offsets of the
// would-be match against the sets the automaton allows there (the set at offset o holds
// exactly the scanned bytes).  Returns the candidate start or kNone.
__device__ __forceinline__ uint64_t pf_candidate(const WalkArgs& a, const PfArgs& pf, const uint32_t* sets, uint64_t q) {
  if (q < pf.o) return kNone;
  const uint64_t s = q - pf.o;
  if (s + 4 > a.n) {  // the last bytes of the buffer: byte loads
    for (uint32_t d = 0; d < pf.n_sets; d++) {
      if (s + d >= a.n) return a.text_continues ? s : kNone;  // a shard's halo ends here: let the automaton report it
      const uint32_t b = a.text[s + d];
      if (!((sets[d * 8 + (b >> 5)] >> (b & 31)) & 1u)) return kNone;
    }
    return s;
  }
  // four bytes at s from two aligned words: one memory round trip
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(a.text + s) & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(a.text + s) & 3) * 8;
  const uint32_t w0 = __ldg(wp), w1 = sh ? __ldg(wp + 1) : 0u;
  const uint32_t w = __funnelshift_r(w0, w1, sh);
  bool ok = true;
#pragma unroll
  for (uint32_t d = 0; d < 4; d++) {
    const uint32_t b = (w >> (8 * d)) & 0xFFu;
    if (d < pf.n_sets) ok = ok && ((sets[d * 8 + (b >> 5)] >> (b & 31)) & 1u);
  }
  return ok ? s : kNone;
}

constexpr uint32_t kPfSlots = 6;  // queued hits per lane between two flushes
constexpr uint32_t kPfWarpSmem = kPfSlots * 32 * 2 + kPfSlots * 32 * 4;  // u16 positions + u32 match lengths

// The chain over chunk k.  Hits are only QUEUED while the chunk streams by (a two-byte push by
// the lane that saw the byte: no warp-wide step per hit); at the end of the chunk every lane
// verifies its own queue -- fingerprint, then the anchored automaton -- with all lanes that
// have work active at once, and the warp then takes the verified matches in position order
// (one warp-wide minimum per match) and applies the find_iter rule to them.
template <int NB, typename Runner>
__device__ __forceinline__ uint64_t pf_walk_chunk(const WalkArgs& a, const PfArgs& pf, const uint32_t* sets, unsigned char* warp_smem,
                                                  const Runner& R, uint64_t k, Chain& c, uint64_t* first_cand, uint64_t* dst,
                                                  uint64_t w_at, uint64_t limit_out) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t cb = a.base + k * (uint64_t)a.chunk;
  const uint64_t ce = min(cb + a.chunk, a.limit);
  const uint64_t q_hi = min(ce, a.n);       // scanned bytes [cb, q_hi)
  uint16_t* qpos = reinterpret_cast<uint16_t*>(warp_smem);                         // [slot][lane]: q - cb
  uint32_t* qlen = reinterpret_cast<uint32_t*>(warp_smem + kPfSlots * 32 * 2);     // [slot][lane]: match length, 0 = none
  uint64_t total = 0, fc = kNone;
  uint64_t p = c.p, lm = c.lm;               // warp-uniform iterator state
  uint32_t cnt = 0;                          // queued hits of this lane
  const bool exact = c.chain;
  uint64_t long_s = kNone;                   // uniform: a match the iterator needs ran past the cap (chunk deferred)
  constexpr uint32_t kLenAgain = 0xFFFFFFFFu, kLenTooLong = 0xFFFFFFFEu;
  auto accept = [&](uint64_t s, uint64_t e) {  // uniform arguments
    if (s < p) return;
    if (fc == kNone) fc = s;
    if (lane == 0 && w_at + total < limit_out) {
      dst[2 * (w_at + total)] = s;
      dst[2 * (w_at + total) + 1] = e;
    }
    total++;
    p = lm = e;
  };
  auto flush = [&]() {
    uint32_t maxc = cnt;
    for (int o = 16; o; o >>= 1) maxc = max(maxc, __shfl_xor_sync(0xffffffffu, maxc, o));
    if (maxc == 0) return;
    for (uint32_t r = 0; r < maxc; r++) {  // round r: every lane with an r-th hit verifies it
      if (r < cnt) {
        const uint64_t q = cb + qpos[r * 32 + lane];
        const uint64_t s = pf_candidate(a, pf, sets, q);  // includes the byte at q itself (the set at offset o)
        uint32_t len = 0;
        if (s != kNone && s >= p) {
          const uint64_t e = pf_verify(&a, &R, s, exact);
          if (e == kTooLong) len = kLenTooLong;
          else if (e != kNone) len = e - s >= kLenTooLong ? kLenAgain : (uint32_t)(e - s);
        }
        qlen[r * 32 + lane] = len;
      }
    }
    __syncwarp();
    // verified matches in position order: each lane offers its first pending one
    uint32_t cur = 0;
    for (;;) {
      while (cur < cnt && qlen[cur * 32 + lane] == 0) cur++;
      const uint32_t key = cur < cnt ? (uint32_t)qpos[cur * 32 + lane] : 0xFFFFFFFFu;
      const uint32_t m = __reduce_min_sync(0xffffffffu, key);
      if (m == 0xFFFFFFFFu) break;
      const int owner = __ffs(__ballot_sync(0xffffffffu, key == m)) - 1;
      const uint32_t len = __shfl_sync(0xffffffffu, cur < cnt ? qlen[cur * 32 + lane] : 0u, owner);
      const uint64_t s = cb + m - pf.o;
      if ((int)lane == owner) cur++;
      if (s < p) continue;  // inside the match accepted before it
      const uint64_t e = len == kLenTooLong ? kTooLong : len == kLenAgain ? pf_verify(&a, &R, s, exact) : s + len;  // (4 GiB or more: ask again)
      if (e == kTooLong) { long_s = s; break; }
      accept(s, e);
    }
    cnt = 0;
    __syncwarp();
  };
  const uint32_t cc[4] = {pf.bcast[0], pf.bcast[1], pf.bcast[2], pf.bcast[3]};
  for (uint64_t off = cb; off < q_hi; off += 2048) {
    uint4 v[4];
    const bool whole = off + 2048 <= q_hi;  // the common piece: every byte inside the chunk and the buffer
    const uint8_t* src = a.text + off + lane * 16;
    if (whole) {
#pragma unroll
      for (int u = 0; u < 4; u++) v[u] = ldg128(src + u * 512);
    } else {
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const uint64_t pos = off + u * 512 + lane * 16;
        if (pos + 16 <= a.n) {
          v[u] = ldg128(a.text + pos);
        } else {  // the last bytes of the buffer
          uint32_t w[4] = {0, 0, 0, 0};
          for (int j = 0; j < 16; j++)
            if (pos + j < a.n) w[j >> 2] |= (uint32_t)a.text[pos + j] << (8 * (j & 3));
          v[u] = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
    const uint32_t cnt_before = cnt;
    const uint32_t rel0 = (uint32_t)(off - cb) + lane * 16;
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const uint32_t t0 = swar_any<NB>(cc, v[u].x), t1 = swar_any<NB>(cc, v[u].y), t2 = swar_any<NB>(cc, v[u].z), t3 = swar_any<NB>(cc, v[u].w);
      if ((t0 | t1 | t2 | t3) != 0) {  // this lane only: queue the flagged bytes (a flag above a true hit may be spurious: flush() looks again)
        uint32_t bits = flags_to_bits(t0) | (flags_to_bits(t1) << 4) | (flags_to_bits(t2) << 8) | (flags_to_bits(t3) << 12);
        const uint32_t rel = rel0 + u * 512;
        if (!whole) {
          const uint64_t pos = cb + rel;
          bits = pos >= q_hi ? 0u : (pos + 16 > q_hi ? bits & ((1u << (uint32_t)(q_hi - pos)) - 1u) : bits);
        }
        while (bits) {
          const int j = __ffs(bits) - 1;
          bits &= bits - 1;
          if (cnt < kPfSlots) qpos[cnt * 32 + lane] = (uint16_t)(rel + j);
          cnt++;
        }
      }
    }
    if (__any_sync(0xffffffffu, cnt > kPfSlots)) {
      // a lane met more of the bytes than it can queue (a haystack full of them): verify what was
      // queued before this piece, then take this piece lane by lane, in order
      cnt = cnt_before;
      flush();
#pragma unroll 1
      for (int u = 0; u < 4; u++) {
        const uint64_t pos = off + u * 512 + lane * 16;
        uint32_t todo = __ballot_sync(0xffffffffu, pos < q_hi);
        while (todo) {
          const int l = __ffs(todo) - 1;
          todo &= todo - 1;
          const uint64_t lpos = __shfl_sync(0xffffffffu, pos, l);
          for (uint32_t j = 0; j < 16 && lpos + j < q_hi; j++) {  // uniform: every lane evaluates lane l's bytes (broadcast loads)
            const uint64_t q = lpos + j;
            const uint32_t byte = __ldg(a.text + q);
            bool is = false;
            for (uint32_t i = 0; i < pf.n_bytes; i++) is = is || byte == (pf.bcast[i] & 0xFFu);
            if (!is) continue;
            const uint64_t s = pf_candidate(a, pf, sets, q);
            if (s == kNone || s < p || long_s != kNone) continue;
            const uint64_t e = pf_verify(&a, &R, s, exact);
            if (e == kTooLong) long_s = s;
            else if (e != kNone) accept(s, e);
          }
        }
      }
    } else if (__any_sync(0xffffffffu, cnt + 2 > kPfSlots)) {
      flush();  // little room left: empty the queues before the next piece
    }
    if (long_s != kNone) break;
  }
  if (long_s == kNone) flush();
  if (long_s != kNone) {  // as chunk_walk: nothing of this walk counts, the stitch walks the chunk again
    if (exact && lane == 0) atomicMin(a.long_req, (unsigned long long)long_s);
    *first_cand = kTooLong;
    return 0;
  }
  c.p = p;
  c.lm = lm;
  if (total) c.chain = true;
  *first_cand = fc;
  return total;
}

template <int FAST, int NB>
__global__ void __launch_bounds__(256, 3) literal_scan(const __grid_constant__ WalkArgs a, const __grid_constant__ PfArgs pf, int mode) {
  const auto R = RunnerSetup<FAST>::make(a);
  __shared__ uint32_t sets[32];
  __shared__ __align__(16) unsigned char queues[8 * kPfWarpSmem];  // blockDim.x == 256
  if (threadIdx.x < 32) sets[threadIdx.x] = pf.sets[threadIdx.x >> 3][threadIdx.x & 7];
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  unsigned char* wq = queues + (threadIdx.x >> 5) * kPfWarpSmem;
  const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  if (mode == 2) {  // sequential pass: one warp, chunk after chunk with exact entry states
    if (warp != 0) return;
    Chain c;
    c.p = a.in_p[a.seq_from];
    c.lm = a.in_lm[a.seq_from];
    c.chain = c.p != kSpec;
    for (uint64_t k = a.seq_from; k < a.n_chunks; k++) {
      const bool spec = !c.chain;
      if (spec) { c.p = 0; c.lm = kNone; }
      else if (lane == 0) { a.in_p[k] = c.p; a.in_lm[k] = c.lm; }
      uint64_t fc = kNone;
      const uint64_t total = pf_walk_chunk<NB>(a, pf, sets, wq, R, k, c, &fc, a.stage, k * (uint64_t)a.stage_cap, (k + 1) * (uint64_t)a.stage_cap);
      if (spec && total == 0) { c.p = a.base + k * (uint64_t)a.chunk + 1; }
      if (lane == 0) finish_chunk(a, k, c, total, fc, spec);
      if (fc == kTooLong) return;  // as walk_sequential
      c.chain = true;
    }
    return;
  }
  const uint64_t work = mode == 1 ? (uint64_t)*a.n_dirty : a.n_chunks;
  for (uint64_t idx = warp; idx < work; idx += n_warps) {
    const uint64_t k = mode == 1 ? a.dirty_list[idx] : idx;
    if (mode == 3 && (a.count[k] <= a.stage_cap)) continue;
    Chain c;
    c.p = a.in_p[k];
    c.lm = a.in_lm[k];
    c.chain = c.p != kSpec;
    const bool spec = !c.chain;
    if (spec) { c.p = 0; c.lm = kNone; }  // accept from the chunk's first candidate on
    uint64_t fc = kNone;
    if (mode == 3) {
      pf_walk_chunk<NB>(a, pf, sets, wq, R, k, c, &fc, a.out, a.offset[k], a.cap);
      continue;
    }
    const uint64_t total = pf_walk_chunk<NB>(a, pf, sets, wq, R, k, c, &fc, a.stage, k * (uint64_t)a.stage_cap, (k + 1) * (uint64_t)a.stage_cap);
    if (spec && total == 0) c.p = a.base + k * (uint64_t)a.chunk + 1;  // what a speculative walk without matches reports (never used: IDENT)
    if (lane == 0) finish_chunk(a, k, c, total, fc, spec);
  }
}
#define RB_INSTANTIATE_LITERAL_SCAN(F, N) \
  template __global__ void literal_scan<F, N>(const __grid_constant__ WalkArgs, const __grid_constant__ PfArgs, int);
RB_INSTANTIATE_LITERAL_SCAN(0, 1) RB_INSTANTIATE_LITERAL_SCAN(0, 2) RB_INSTANTIATE_LITERAL_SCAN(0, 3) RB_INSTANTIATE_LITERAL_SCAN(0, 4)
RB_INSTANTIATE_LITERAL_SCAN(1, 1) RB_INSTANTIATE_LITERAL_SCAN(1, 2) RB_INSTANTIATE_LITERAL_SCAN(1, 3) RB_INSTANTIATE_LITERAL_SCAN(1, 4)

// compact_spans without the re-walk of overflowed chunks (literal_scan mode 3 does those)
__global__ void __launch_bounds__(256) compact_staged(WalkArgs a) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp0 = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  const ulonglong2* stage = reinterpret_cast<const ulonglong2*>(a.stage);
  ulonglong2* dst = reinterpret_cast<ulonglong2*>(a.out);
  for (uint64_t g = warp0; g * 32 < a.n_chunks; g += n_warps) {
    const uint64_t k = g * 32 + lane;
    const uint64_t my_cnt = k < a.n_chunks ? a.count[k] : 0;
    const uint64_t my_at = k < a.n_chunks ? a.offset[k] : 0;
    const uint32_t my_skip = k < a.n_chunks ? a.skip[k] : 0;
    uint32_t todo = __ballot_sync(0xffffffffu, my_cnt != 0 && my_cnt <= a.stage_cap);
    while (todo) {
      const int j = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint64_t cnt = __shfl_sync(0xffffffffu, my_cnt, j), at = __shfl_sync(0xffffffffu, my_at, j);
      const uint32_t sk = __shfl_sync(0xffffffffu, my_skip, j);
      for (uint64_t i = lane; i < cnt; i += 32)
        if (at + i < a.cap) dst[at + i] = stage[(g * 32 + j) * (uint64_t)a.stage_cap + sk + i];
    }
  }
}

// FUSED: each lane also walks the find_iter chain over its own segment right after
// scanning it (chunk == segment), while the segment's haystack bytes are still in L2 and
// without a second kernel's bitmap round trip.  The walk is speculative exactly like
// walk_chunks; stitch_check / walk_chunks(dirty) / compact_spans finish the job.
// Haystack bytes reach shared memory by TMA.  When a warp's 32 lanes own 32 consecutive
// full segments, the haystack is addressed as a 2-D tensor [rows = segments][cols = bytes]
// and ONE elected lane issues four [16 B x 32 rows] box loads per 64-byte group for the
// whole warp (per-lane 64-byte bulk copies were TMA-issue bound: a third of all issued
// instructions were mbarrier polls).  Ragged ends and redo lists use per-lane bulk copies.
// One 64-byte group on the full class-indexed table (global memory), highest address
// first: the path a lane of scan_rev_fast takes while it is outside the hot set.
__device__ __noinline__ uint32_t slow_group(const uint16_t* trans, const uint8_t* classes, uint32_t stride, uint32_t match_lo, uint32_t s,
                                            uint4 c0, uint4 c1, uint4 c2, uint4 c3, uint64_t* bits_out) {
  const uint32_t w[16] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w, c3.x, c3.y, c3.z, c3.w};
  uint64_t bits = 0;
  for (int j = 63; j >= 0; j--) {
    const uint32_t byte = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
    s = trans[s * stride + classes[byte]];
    if (s >= match_lo) bits |= 1ull << j;
  }
  *bits_out = bits;
  return s;
}

template <int FUSED>
__global__ void __launch_bounds__(1024, 1) scan_rev_fast(ScanArgs a, WalkArgs wa, const __grid_constant__ CUtensorMap tmap) {
  // shared layout: 512-byte aligned, per warp 2 stages x 32 lanes x 64 B, then the mbarriers, then
  // [reverse hot table][forward hot table (FUSED == 1)].  The rings come first so that their
  // addresses depend on nothing but the warp index: behind the tables they were recomputed from
  // the table sizes in every 64-byte group (the kernel has no registers to spare).
  // (the reverse table uses signed row ids: match rows below tbase, see hot_stage_signed)
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t rings = ((uint32_t)__cvta_generic_to_shared(g_smem) + 511u) & ~511u;
  const uint32_t ring = rings + wid * kRingWarpBytes;
  const uint32_t bar0 = rings + (blockDim.x >> 5) * kRingWarpBytes + wid * kRingBarBytes;
  const uint32_t tbase = rings + a.tbase_off;  // = rings + warps * (ring + barriers) + hot_signed_below(a.hot), a multiple of 256
  const uint32_t fbase = rings + a.fbase_off;  // = ... + hot_signed_bytes(a.hot)
  const uint32_t rml = a.hot.match_lo;
  {
    hot_stage_signed(a.hot, tbase);
    if (FUSED == 1) hot_stage(wa.fwd_hot, fbase);
    if (lane == 0) {
      mbar_init(bar0, 32);
      mbar_init(bar0 + 8, 32);
      for (uint32_t sidx = 0; sidx < kBoxStages; sidx++) mbar_init(bar0 + 16 + 8 * sidx, 1);  // boxed (2-D TMA) mode: one elected lane arrives for the warp
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  const uint32_t my_slot = ring + lane * kRingLaneStride;  // + stage * kRingStageBytes
  const uint64_t total = a.redo_list ? (uint64_t)*a.n_redo : a.n_seg;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t first = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint64_t rounds = (total + stride - 1) / stride;  // uniform: every warp makes every round
  uint32_t uses = 0;  // ring uses so far (same for the whole warp): stage = uses & 1, parity = (uses >> 1) & 1
  uint32_t slot_b = 0, par_b = 0;  // boxed mode: ring slot and barrier parity of the next group to consume
  for (uint64_t round = 0; round < rounds; round++) {
    const uint64_t idx = first + round * stride;
    const bool live = idx < total;
    uint64_t t = 0, lo = 0, hi = 0, i = 0;
    uint32_t e = 0;
    uint32_t cold = 0;  // != 0: the lane is outside the hot set, in this state of the full table (e sits in the trap row)
    auto enter = [&](uint32_t full) {  // e is a signed row id (hot_sid)
      const uint32_t h = a.hot.full2hot[full];
      if (h != 0xFFFFu) { e = hot_sid(h, rml); cold = 0; }
      else { e = 1; cold = full; }
    };
    auto full_state = [&]() -> uint32_t { return cold ? cold : a.hot.hot2full[hot_idx(e, rml)]; };
    auto full_step = [&](uint32_t s, uint32_t byte) -> uint32_t { return a.dfa.trans[s * a.dfa.stride + a.dfa.classes[byte]]; };
    // one 64-byte group: table steps in shared memory; a lane that ends in the trap row
    // (it met a byte outside the hot set, or was cold already) redoes the group on the full table
    auto do_group = [&](const uint4& c0, const uint4& c1, const uint4& c2, const uint4& c3, bool rec, uint32_t& bhi, uint32_t& blo) {
      const uint32_t e0 = e;
      bhi = blo = 0;
      rev_block16_s(tbase, c3, e, bhi);
      rev_block16_s(tbase, c2, e, bhi);
      rev_block16_s(tbase, c1, e, blo);
      rev_block16_s(tbase, c0, e, blo);
      if (!rec) bhi = blo = 0;  // warm-up bytes: states only
      if (e == 1u) {
        uint64_t bits;
        const uint32_t s1 = slow_group(a.dfa.trans, a.dfa.classes, a.dfa.stride, a.dfa.match_lo,
                                       cold ? cold : a.hot.hot2full[hot_idx(e0, rml)], c0, c1, c2, c3, &bits);
        bhi = rec ? (uint32_t)(bits >> 32) : 0u;
        blo = rec ? (uint32_t)bits : 0u;
        enter(s1);
      }
    };
    // the same for a group that sits in a ring slot (swizzled, boxed mode): 16 bytes are fetched right
    // before their turn, so that 8 registers hold haystack bytes instead of 16 (the kernel lives on 64
    // registers and was recomputing its ring addresses in every group for lack of them); the rare
    // trap-row exit reads the slot again
    auto do_group_slot = [&](uint32_t b, uint32_t sw, bool rec, uint32_t& bhi, uint32_t& blo) {
      const uint32_t e0 = e;
      bhi = blo = 0;
      uint4 x = lds128(b + (48u ^ sw)), y = lds128(b + (32u ^ sw));
      rev_block16_s(tbase, x, e, bhi);
      x = lds128(b + (16u ^ sw));
      rev_block16_s(tbase, y, e, bhi);
      y = lds128(b + (0u ^ sw));
      rev_block16_s(tbase, x, e, blo);
      rev_block16_s(tbase, y, e, blo);
      if (!rec) bhi = blo = 0;
      if (e == 1u) {
        const uint4 c0 = lds128(b + (0u ^ sw)), c1 = lds128(b + (16u ^ sw)), c2 = lds128(b + (32u ^ sw)), c3 = lds128(b + (48u ^ sw));
        uint64_t bits;
        const uint32_t s1 = slow_group(a.dfa.trans, a.dfa.classes, a.dfa.stride, a.dfa.match_lo,
                                       cold ? cold : a.hot.hot2full[hot_idx(e0, rml)], c0, c1, c2, c3, &bits);
        bhi = rec ? (uint32_t)(bits >> 32) : 0u;
        blo = rec ? (uint32_t)bits : 0u;
        enter(s1);
      }
    };
    if (live) {
      t = a.redo_list ? a.redo_list[idx] : idx;
      lo = min(a.base + t * a.seg, a.limit);  // multiple of 64 (or limit)
      hi = min(lo + a.seg, a.limit);          // multiple of 64 (or limit == n)
      i = hi;
      if (a.redo_list) {
        enter(a.fin[t + 1]);
      } else {
        i = min(hi + a.warm, a.n);
        uint32_t s = pick_start_rev(a.dfa, a.text, a.n, i);
        // ragged top of the warm-up (only next to the end of the haystack): full table, byte by byte
        while (i > hi && (i & 63)) { i--; s = full_step(s, a.text[i]); }
        enter(s);
      }
      if (i == hi) {
        a.guess[t] = (uint16_t)full_state();
        if (i & 63) {  // ragged top of the segment itself (last segment only)
          uint64_t word = 0;
          uint32_t s = full_state();
          while (i > lo && (i & 63)) {
            i--;
            s = full_step(s, a.text[i]);
            if (s >= a.dfa.match_lo) word |= 1ull << (i & 63);
          }
          a.bitmap[i >> 6] = word;
          enter(s);
        }
      }
    }
    // bytes [lo, i) remain, i a multiple of 64: whole groups through the ring
    const uint32_t my_groups = live ? (uint32_t)((i - lo) >> 6) : 0;
    uint32_t max_groups = my_groups;
    for (int o = 16; o; o >>= 1) max_groups = max(max_groups, __shfl_xor_sync(0xffffffffu, max_groups, o));
    const uint8_t* top = a.text + i;  // group k covers [top - 64(k+1), top - 64k)
    // 2-D path: whole warp live, no redo list, identical geometry in every lane
    // (full segments, full warm-up), and all rows (incl. the warm-up row) inside the map.
    const uint64_t t0 = __shfl_sync(0xffffffffu, t, 0);
    const bool uniform = live && !a.redo_list && hi - lo == a.seg && i == hi + a.warm && t == t0 + lane;
    const bool all_uniform = __all_sync(0xffffffffu, uniform) && a.warm <= a.seg;
    const bool boxed = a.tmap_rows != 0 && all_uniform && t0 + 33 <= a.tmap_rows;
    uint64_t nz = 0;  // FUSED: which bitmap words of this segment are non-zero
    if (boxed) {
      // Tight loop for the common geometry: every lane scans one full segment plus the
      // warm-up, so group counts, the warm-up/record split and the ring slots are warp
      // uniform and one lane drives the TMA for all 32.
      const uint32_t n_groups = (a.seg + a.warm) >> 6, n_warm = a.warm >> 6;
      const uint32_t barb = bar0 + 16;
      auto issue_box = [&](uint32_t k, uint32_t slot) {  // lane 0 only
        const uint32_t bar = barb + slot * 8;
        mbar_arrive_tx(bar, 2048);
        // byte offset of the group inside row-space: segment bytes then the neighbour row's warm-up bytes
        const uint32_t o = a.seg + a.warm - 64u * (k + 1);
        const uint32_t row = (uint32_t)t0 + (o >= a.seg ? 1u : 0u);
        const uint32_t col = o >= a.seg ? o - a.seg : o;
        tma_box(ring + slot * kRingStageBytes, &tmap, col, row, bar);
      };
      if (lane == 0) {
#pragma unroll
        for (uint32_t j = 0; j < kBoxStages; j++)
          if (j < n_groups) issue_box(j, (slot_b + j) % kBoxStages);
      }
      uint64_t* bw = a.bitmap + (hi >> 6);
      uint64_t pw1 = 0, pw2 = 0, pw3 = 0;  // the previous three words (higher addresses) of the current sector
      const bool sector_stores = (a.seg & 255u) == 0;  // one past the segment's last bitmap word
      // the box lands row-major (row = lane, 64 bytes) with the 64B swizzle: 16-byte chunk j of
      // row r sits at chunk j ^ ((r >> 1) & 3), which makes the four LDS.128 conflict-free
      const uint32_t my_b = ring + lane * 64u;
      const uint32_t sw = ((lane >> 1) & 3u) << 4;
      for (uint32_t k = 0; k < n_groups; k++) {
        mbar_wait(barb + slot_b * 8, par_b);
        const uint32_t b = my_b + slot_b * kRingStageBytes;
        if (k == n_warm) a.guess[t] = (uint16_t)full_state();
        const bool rec = k >= n_warm;
        uint32_t bhi, blo;
        do_group_slot(b, sw, rec, bhi, blo);
        if (rec) {
          // Bitmap words leave as whole 32-byte sectors (four words, every fourth group):
          // an 8-byte store per group is a partial-sector write from each lane, and those
          // capped the whole kernel at 3.0 TB/s (5.0 TB/s with the stores removed).
          const uint64_t wv = ((uint64_t)bhi << 32) | blo;
          --bw;
          if (!sector_stores) *bw = wv;
          else if (((k - n_warm) & 3u) == 3u) st_sector(bw, wv, pw1, pw2, pw3);
          pw3 = pw2; pw2 = pw1; pw1 = wv;
          if (FUSED) nz = (nz << 1) | ((bhi | blo) ? 1ull : 0ull);
        }
        // every lane has its 64 bytes in registers: lane 0 refills the slot kBoxStages groups ahead
        __syncwarp();
        if (lane == 0 && k + kBoxStages < n_groups) issue_box(k + kBoxStages, slot_b);
        if (++slot_b == kBoxStages) { slot_b = 0; par_b ^= 1; }
      }
    } else {
    auto issue = [&](uint32_t k) {    // every lane arrives; lanes with data also copy
      const uint32_t u = uses + k;
      const uint32_t bar = bar0 + (u & 1) * 8;
      if (k < my_groups) {
        mbar_arrive_tx(bar, 64);
        bulk_g2s(my_slot + (u & 1) * kRingStageBytes, top - 64ull * (k + 1), 64, bar);
      } else {
        mbar_arrive_tx(bar, 0);
      }
    };
    if (max_groups > 0) issue(0);
    if (max_groups > 1) issue(1);
    for (uint32_t k = 0; k < max_groups; k++) {
      const uint32_t u = uses + k;
      const uint32_t slot = my_slot + (u & 1) * kRingStageBytes;
      mbar_wait(bar0 + (u & 1) * 8, (u >> 1) & 1);
      if (k < my_groups) {
        const uint4 c0 = lds128(slot), c1 = lds128(slot + 16), c2 = lds128(slot + 32), c3 = lds128(slot + 48);
        const uint64_t g = i - 64ull * (k + 1);  // first byte of this group
        if (g + 64 == hi) a.guess[t] = (uint16_t)full_state();
        uint32_t bhi, blo;
        do_group(c0, c1, c2, c3, g < hi, bhi, blo);
        if (g < hi) {
          a.bitmap[g >> 6] = ((uint64_t)bhi << 32) | blo;
          if (FUSED && (bhi | blo)) nz |= 1ull << (((g - lo) >> 6) & 63);
        }
      }
      // the slot's bytes have been consumed: refill it for the group after next
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (k + 2 < max_groups) issue(k + 2);
    }
    uses += max_groups;
    }
    if (live) {
      const uint32_t s_lo = full_state();
      a.fin[t] = (uint16_t)s_lo;
      if (lo == 0) *a.flag0 = a.dfa.trans[s_lo * a.dfa.stride + a.dfa.stride - 1] >= a.dfa.match_lo;
      if (FUSED) {
        typename RunnerSetup<FUSED == 2 ? 2 : 1>::type R;
        if constexpr (FUSED == 2) {
          R.len = wa.fixed_len;
        } else {
          R.tb = fbase;
          R.thr = wa.fwd_hot.match_lo;
          R.start_e = wa.fwd_hot.start;
          R.eof = wa.fwd_hot.eof;
          R.match_lo = wa.fwd.match_lo;
        }
        Chain c;
        c.p = wa.in_p[t];
        c.lm = wa.in_lm[t];
        c.chain = c.p != kSpec;
        const bool spec = !c.chain;
        if (spec) { c.p = wa.base + t * (uint64_t)wa.chunk + 1; c.lm = kNone; }
        uint64_t fc = kNone, total = 0;
        // segments longer than 64 words, the ragged last segment and position 0 fall back to "unknown"
        const bool nz_ok = a.seg <= 4096 && !(hi & 63) && lo != 0;
        const uint32_t walkers = __ballot_sync(__activemask(), c.p != kNone);
        if (c.p != kNone)
          total = chunk_walk(wa, R, t, c, &fc, wa.stage, t * (uint64_t)wa.stage_cap, (t + 1) * (uint64_t)wa.stage_cap, nz_ok ? nz : ~0ull, walkers);
        finish_chunk(wa, t, c, total, fc, spec);
      }
    }
  }
}
template __global__ void scan_rev_fast<0>(ScanArgs, WalkArgs, const __grid_constant__ CUtensorMap);
template __global__ void scan_rev_fast<1>(ScanArgs, WalkArgs, const __grid_constant__ CUtensorMap);
template __global__ void scan_rev_fast<2>(ScanArgs, WalkArgs, const __grid_constant__ CUtensorMap);




// ------------------------------------------------------------- scan_fwd_fast --
// Forward counterpart of scan_rev_fast for whole-haystack is_match / shortest_match:
// hot table in shared memory, the haystack through the 2-D TMA ring, per segment the first
// match END (positions as in scan_fwd_reduce), the state assumed at the segment's first
// byte (guess) and the exact state after its last (fin).  It takes the warps of 32
// consecutive full segments [skip_lo, skip_hi); scan_fwd_reduce does the ragged edges, the
// EOF step and the redo rounds.
template <int BIT0>
__device__ __forceinline__ void fwd_word(uint32_t tb, uint32_t w, uint32_t& e, uint32_t& bits, uint32_t thr) {
  e = hot_next<0>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 0);
  e = hot_next<1>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 1);
  e = hot_next<2>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 2);
  e = hot_next<3>(tb, w, e); if (e >= thr) bits |= 1u << (BIT0 + 3);
}
template <int BIT0>
__device__ __forceinline__ void fwd_block16(uint32_t tb, const uint4& v, uint32_t& e, uint32_t& bits, uint32_t thr) {
  fwd_word<BIT0 + 0>(tb, v.x, e, bits, thr);
  fwd_word<BIT0 + 4>(tb, v.y, e, bits, thr);
  fwd_word<BIT0 + 8>(tb, v.z, e, bits, thr);
  fwd_word<BIT0 + 12>(tb, v.w, e, bits, thr);
}
__device__ __noinline__ uint32_t slow_group_fwd(const uint16_t* trans, const uint8_t* classes, uint32_t stride, uint32_t match_lo, uint32_t s,
                                                uint4 c0, uint4 c1, uint4 c2, uint4 c3, uint64_t* bits_out) {
  const uint32_t w[16] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w, c3.x, c3.y, c3.z, c3.w};
  uint64_t bits = 0;
  for (int j = 0; j < 64; j++) {
    const uint32_t byte = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
    s = trans[s * stride + classes[byte]];
    if (s >= match_lo) bits |= 1ull << j;
  }
  *bits_out = bits;
  return s;
}
// One group again on the full table, OR-ing the pattern masks of the match states it enters.
__device__ __noinline__ void slow_group_masks(const uint16_t* trans, const uint8_t* classes, const uint64_t* masks, uint32_t stride,
                                              uint32_t match_lo, uint32_t mw, uint32_t s, uint4 c0, uint4 c1, uint4 c2, uint4 c3, uint64_t* acc) {
  const uint32_t w[16] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w, c3.x, c3.y, c3.z, c3.w};
  uint32_t last = 0;
  for (int j = 0; j < 64; j++) {
    const uint32_t byte = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
    s = trans[s * stride + classes[byte]];
    if (s >= match_lo && s != last) {
      last = s;
      for (uint32_t i = 0; i < mw; i++) acc[i] |= masks[(uint64_t)s * mw + i];
    }
  }
}
__global__ void __launch_bounds__(1024, 1) scan_fwd_fast(ScanArgs a, const __grid_constant__ CUtensorMap tmap) {
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t rings = ((uint32_t)__cvta_generic_to_shared(g_smem) + 511u) & ~511u;  // as scan_rev_fast: rings, mbarriers, table
  const uint32_t ring = rings + wid * kRingWarpBytes;
  const uint32_t barb = rings + (blockDim.x >> 5) * kRingWarpBytes + wid * kRingBarBytes;
  const uint32_t tbase = rings + (blockDim.x >> 5) * (kRingWarpBytes + kRingBarBytes);
  hot_stage(a.hot, tbase);
  if (lane == 0) {
    for (uint32_t sidx = 0; sidx < kBoxStages; sidx++) mbar_init(barb + 8 * sidx, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t thr = a.hot.match_lo;
  const uint32_t n_groups = (a.seg + a.warm) >> 6, n_warm = a.warm >> 6;
  const uint64_t n_warps = (a.skip_hi - a.skip_lo) >> 5;
  const uint64_t warp0 = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t warp_stride = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  uint32_t slot_b = 0, par_b = 0;
  const uint32_t my_b = ring + lane * 64u;
  const uint32_t sw = ((lane >> 1) & 3u) << 4;
  for (uint64_t wq = warp0; wq < n_warps; wq += warp_stride) {
    const uint64_t t0 = a.skip_lo + wq * 32, t = t0 + lane;
    const uint64_t lo = a.base + t * a.seg;  // this lane scans [lo - warm, lo) unrecorded, then [lo, lo + seg)
    uint32_t e, cold = 0;
    auto enter = [&](uint32_t full) {
      const uint32_t h = a.hot.full2hot[full];
      if (h != 0xFFFFu) { e = h; cold = 0; }
      else { e = 1; cold = full; }
    };
    auto full_state = [&]() -> uint32_t { return cold ? cold : a.hot.hot2full[e]; };
    enter(pick_start_fwd(a.dfa, a.text, a.n, lo - a.warm));
    auto issue_box = [&](uint32_t k, uint32_t slot) {  // lane 0 only
      const uint32_t bar = barb + slot * 8;
      mbar_arrive_tx(bar, 2048);
      // row-space offset of group k relative to row t0: the warm-up groups lie at the end of the previous row
      const uint32_t o = 64u * k;
      const bool prev = o < a.warm;
      const uint32_t row = (uint32_t)(t0 - a.skip_lo) + (prev ? 0u : 1u);  // tensor row 0 = segment skip_lo - 1
      const uint32_t col = prev ? a.seg - a.warm + o : o - a.warm;
      tma_box(ring + slot * kRingStageBytes, &tmap, col, row, bar);
    };
    if (lane == 0) {
#pragma unroll
      for (uint32_t j = 0; j < kBoxStages; j++)
        if (j < n_groups) issue_box(j, (slot_b + j) % kBoxStages);
    }
    uint64_t first = kNone;
    uint64_t acc[kMaxMaskWords] = {0, 0, 0, 0};
    for (uint32_t k = 0; k < n_groups; k++) {
      mbar_wait(barb + slot_b * 8, par_b);
      const uint32_t b = my_b + slot_b * kRingStageBytes;
      const uint4 c0 = lds128(b + (0u ^ sw)), c1 = lds128(b + (16u ^ sw)), c2 = lds128(b + (32u ^ sw)), c3 = lds128(b + (48u ^ sw));
      if (k == n_warm) a.guess[t] = (uint16_t)full_state();
      const bool rec = k >= n_warm;
      const uint32_t e0 = e, cold0 = cold;
      const uint32_t th = rec ? thr : 0xFFFFFFFFu;
      uint32_t blo = 0, bhi = 0;
      fwd_block16<0>(tbase, c0, e, blo, th);
      fwd_block16<16>(tbase, c1, e, blo, th);
      fwd_block16<0>(tbase, c2, e, bhi, th);
      fwd_block16<16>(tbase, c3, e, bhi, th);
      if (e == 1u) {  // left the hot set (or was cold): redo the group on the full table
        uint64_t bits;
        const uint32_t s1 = slow_group_fwd(a.dfa.trans, a.dfa.classes, a.dfa.stride, a.dfa.match_lo, cold ? cold : a.hot.hot2full[e0],
                                           c0, c1, c2, c3, &bits);
        bhi = rec ? (uint32_t)(bits >> 32) : 0u;
        blo = rec ? (uint32_t)bits : 0u;
        enter(s1);
      }
      if (first == kNone && (bhi | blo)) {
        const uint64_t bits = ((uint64_t)bhi << 32) | blo;
        first = lo + 64ull * (k - n_warm) + (uint64_t)(__ffsll((long long)bits) - 1);
      }
      if (a.seg_mask && (bhi | blo))  // RegexSet: a match state was entered in this group (rare on this path): which patterns?
        slow_group_masks(a.dfa.trans, a.dfa.classes, a.dfa.masks, a.dfa.stride, a.dfa.match_lo, a.dfa.mask_words,
                         cold0 ? cold0 : a.hot.hot2full[e0], c0, c1, c2, c3, acc);
      __syncwarp();
      if (lane == 0 && k + kBoxStages < n_groups) issue_box(k + kBoxStages, slot_b);
      if (++slot_b == kBoxStages) { slot_b = 0; par_b ^= 1; }
    }
    a.fin[t] = (uint16_t)full_state();
    a.seg_first[t] = first;
    if (a.seg_mask)
      for (uint32_t w = 0; w < a.dfa.mask_words; w++) a.seg_mask[t * a.dfa.mask_words + w] = acc[w];
  }
}

__global__ void init_walk_entries(uint64_t* in_p, uint64_t* in_lm, uint32_t* skip, uint64_t n_chunks, uint64_t p0, uint64_t lm0) {
  for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < n_chunks; k += (uint64_t)gridDim.x * blockDim.x) {
    in_p[k] = k == 0 ? p0 : kSpec;
    in_lm[k] = k == 0 ? lm0 : kNone;
    skip[k] = 0;
  }
}

// ----------------------------------------------------------------- stitch ------
// Bring the speculative chunk walks into agreement with the sequential iterator
// (src/re_trait.rs:197-220).  tests/stitch_model.py is the CPU model of this section.
//
// A chunk's true entry state is the exit state of the last chunk to its left that
// CONTRIBUTES: not IDENT (no candidate bit at all -- the iterator passes through, so the
// chunk hands on what it received, not the first position it assumed) and not COVERED
// (the iterator jumps over it).  That is an exclusive prefix "max by p, later chunk wins
// ties" (entries_local / entries_blocks); stitch_resolve then decides per chunk:
//   - entry beyond the chunk                       -> COVERED, contributes no spans
//   - speculative walk, entry before the chunk     -> keep; with look-arounds the START of the
//     first span is re-derived by the reverse-on-slice rule from the true entry
//     (src/exec.rs:651-657, SURVEY hazard H1) and the chunk is walked again only if that
//     changes whether the span is empty (or the reverse scan fails: the iteration stops)
//   - speculative walk entered late, pattern without empty matches / look-arounds -> the real
//     chain and the speculative one meet at the first staged span that starts at or after the
//     entry, provided the span before it had ended by then: drop the spans before it
//   - anything else -> walk again from the exact entry (dirty list)
// Rounds repeat until nothing changes; the leftmost wrong chunk is right after each round.
__device__ __forceinline__ uint64_t chain_key(uint64_t p) { return p == kNone ? ~0ull : p + 1; }
__device__ __forceinline__ uint64_t key_pos(uint64_t key) { return key == ~0ull ? kNone : key - 1; }
__device__ __forceinline__ ChainKey key_join(const ChainKey& left, const ChainKey& right) {  // associative
  return right.key != 0 && right.key >= left.key ? right : left;
}
__device__ __forceinline__ ChainKey chunk_contribution(const WalkArgs& a, uint64_t k) {
  ChainKey c{0, kNone};
  const uint32_t st = a.meta[k] >> 30;
  if (st == kChunkOk || (k == 0 && a.in_p[0] != kSpec)) { c.key = chain_key(a.out_p[k]); c.lm = a.out_lm[k]; }
  return c;
}
// Drop staged spans in front of tp (see above).  Returns false when the chunk must be walked again.
__device__ __forceinline__ bool trim_staged(const WalkArgs& a, uint64_t k, uint64_t tp, uint32_t cnt, uint32_t* skip_out) {
  if (cnt > a.stage_cap) return false;
  const ulonglong2* sp = reinterpret_cast<const ulonglong2*>(a.stage) + k * (uint64_t)a.stage_cap;
  uint32_t lo = 0, hi = cnt;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (sp[mid].x < tp) lo = mid + 1; else hi = mid;
  }
  if (lo != 0 && sp[lo - 1].y > tp) return false;
  *skip_out = lo;
  return true;
}

// Patterns without empty matches / look-arounds, first pass: every chunk looks at its left
// neighbour only.  Exact unless some exit reaches past the following chunk or a chunk lost
// all its spans (counters[2] asks for the general loop then; nothing is lost, the loop
// decides everything again).
__global__ void stitch_fast(WalkArgs a, uint32_t* counters) {
  for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < a.n_chunks;
       k += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t meta = a.meta[k];
    const uint64_t cb = a.base + k * (uint64_t)a.chunk;
    const uint64_t ce_next = min(cb + 2 * (uint64_t)a.chunk, a.limit);
    if ((meta >> 30) == kChunkDeferred) counters[2] = 1;
    if ((meta >> 30) == kChunkOk && k + 1 < a.n_chunks && a.out_p[k] > ce_next) counters[2] = 1;  // a match longer than a chunk
    if (k == 0 || (meta >> 30) != kChunkOk) continue;
    if ((a.meta[k - 1] >> 30) != kChunkOk) continue;  // the neighbour holds no candidate: the entry cannot lie inside this chunk
    const uint64_t tp = a.out_p[k - 1];
    if (tp <= a.first_cand[k]) continue;
    uint32_t lo;
    const uint32_t cnt = meta & kMetaCount;
    if (tp == kNone || !trim_staged(a, k, tp, cnt, &lo) || lo == cnt) { counters[2] = 1; continue; }
    a.skip[k] = lo;
    a.count[k] = cnt - lo;
  }
}

// Exclusive scan of the chunk contributions inside blocks of blockDim.x chunks.
__global__ void entries_local(WalkArgs a, ChainKey* excl, ChainKey* block_tot, uint32_t* first_deferred) {
  __shared__ ChainKey ws[32];
  const uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  ChainKey mine = k < a.n_chunks ? chunk_contribution(a, k) : ChainKey{0, kNone};
  if (k < a.n_chunks && (a.meta[k] >> 30) == kChunkDeferred) atomicMin(first_deferred, (uint32_t)k);
  ChainKey x = mine;
  for (int o = 1; o < 32; o <<= 1) {
    ChainKey y{__shfl_up_sync(0xffffffffu, x.key, o), __shfl_up_sync(0xffffffffu, x.lm, o)};
    if (lane >= o) x = key_join(y, x);
  }
  if (lane == 31) ws[wid] = x;
  __syncthreads();
  if (wid == 0) {
    ChainKey w = lane < (int)(blockDim.x >> 5) ? ws[lane] : ChainKey{0, kNone};
    for (int o = 1; o < 32; o <<= 1) {
      ChainKey y{__shfl_up_sync(0xffffffffu, w.key, o), __shfl_up_sync(0xffffffffu, w.lm, o)};
      if (lane >= o) w = key_join(y, w);
    }
    ws[lane] = w;  // inclusive over warps
  }
  __syncthreads();
  // exclusive value of this thread = (warps before) join (lanes before)
  ChainKey before{__shfl_up_sync(0xffffffffu, x.key, 1), __shfl_up_sync(0xffffffffu, x.lm, 1)};
  if (lane == 0) before = ChainKey{0, kNone};
  if (wid) before = key_join(ws[wid - 1], before);
  if (k < a.n_chunks) excl[k] = before;
  if (threadIdx.x == blockDim.x - 1) block_tot[blockIdx.x] = ws[(blockDim.x >> 5) - 1];
}
// block_tot[b] := join of the blocks before b (exclusive); *grand = join of all blocks.
__global__ void entries_blocks(ChainKey* block_tot, uint64_t n_blocks, ChainKey* grand) {
  __shared__ ChainKey ws[32];
  __shared__ ChainKey carry_s;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = ChainKey{0, kNone};
  __syncthreads();
  for (uint64_t base = 0; base < n_blocks; base += blockDim.x) {
    const uint64_t i = base + threadIdx.x;
    const ChainKey mine = i < n_blocks ? block_tot[i] : ChainKey{0, kNone};
    ChainKey x = mine;
    for (int o = 1; o < 32; o <<= 1) {
      ChainKey y{__shfl_up_sync(0xffffffffu, x.key, o), __shfl_up_sync(0xffffffffu, x.lm, o)};
      if (lane >= o) x = key_join(y, x);
    }
    if (lane == 31) ws[wid] = x;
    __syncthreads();
    if (wid == 0) {
      ChainKey w = lane < (int)(blockDim.x >> 5) ? ws[lane] : ChainKey{0, kNone};
      for (int o = 1; o < 32; o <<= 1) {
        ChainKey y{__shfl_up_sync(0xffffffffu, w.key, o), __shfl_up_sync(0xffffffffu, w.lm, o)};
        if (lane >= o) w = key_join(y, w);
      }
      ws[lane] = w;
    }
    __syncthreads();
    ChainKey before{__shfl_up_sync(0xffffffffu, x.key, 1), __shfl_up_sync(0xffffffffu, x.lm, 1)};
    if (lane == 0) before = ChainKey{0, kNone};
    if (wid) before = key_join(ws[wid - 1], before);
    const ChainKey carry = carry_s;
    if (i < n_blocks) block_tot[i] = key_join(carry, before);
    __syncthreads();
    if (threadIdx.x == 0) carry_s = key_join(carry, ws[(blockDim.x >> 5) - 1]);
    __syncthreads();
  }
  if (threadIdx.x == 0) *grand = carry_s;
}

__global__ void stitch_resolve(WalkArgs a, const ChainKey* excl, const ChainKey* block_tot, uint32_t* counters) {
  const bool strict = a.emulate_slice || a.can_match_empty;
  const uint64_t deferred_hi = (uint64_t)counters[12] + kDeferredWindow;  // counters[12]: entries_local's leftmost deferred chunk
  for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < a.n_chunks;
       k += (uint64_t)gridDim.x * blockDim.x) {
    if (k == 0) {  // chunk 0 holds the real entry state; it is walked again only after a long run was handed to the host
      if ((a.meta[0] >> 30) == kChunkDeferred) { a.dirty_list[atomicAdd(&counters[0], 1u)] = 0; atomicMin(&counters[3], 0u); }
      continue;
    }
    const uint32_t meta = a.meta[k];
    const uint32_t state = meta >> 30, cnt = meta & kMetaCount;
    if (state == kChunkIdent) continue;
    const ChainKey t = key_join(block_tot[k >> 10], excl[k]);  // entries_local runs with 1024 threads per block
    const bool spec = a.in_p[k] == kSpec;
    if (t.key == 0) {  // nothing to the left contributes (a shard entered speculatively): the chunk's own speculation stands
      const uint64_t own_first = a.base + k * (uint64_t)a.chunk + 1;
      const bool as_is = spec ? (state == kChunkOk && a.skip[k] == 0 && !(meta & kMetaPatched))
                              : (state == kChunkOk && a.in_p[k] == own_first && a.in_lm[k] == kNone);  // a deferred chunk walked again without the cap
      if (state == kChunkDeferred && k >= deferred_hi) continue;  // waits for the deferred chunks further left
      if (!as_is) {
        a.dirty_list[atomicAdd(&counters[0], 1u)] = (uint32_t)k;
        a.in_p[k] = state == kChunkDeferred ? own_first : kSpec;
        a.in_lm[k] = kNone;
        atomicMin(&counters[3], (uint32_t)k);
      }
      continue;
    }
    const uint64_t tp = key_pos(t.key), tl = t.lm;
    const uint64_t cb = a.base + k * (uint64_t)a.chunk;
    const uint64_t ce = min(cb + a.chunk, a.limit), c_first = cb + 1;
    uint32_t new_state = kChunkOk, new_skip = 0;
    uint64_t new_count = cnt;
    bool rewalk = false;
    if (tp == kNone || tp > ce) {
      new_state = kChunkCovered;
      new_count = 0;
    } else if (state == kChunkDeferred && k >= deferred_hi) {
      continue;  // waits for the deferred chunks further left (most likely one of their matches covers it)
    } else if (spec && state == kChunkDeferred) {
      rewalk = true;
    } else if (spec) {
      if (strict) {
        bool ok = tp < c_first || (tp == c_first && !a.emulate_slice && !(a.can_match_empty && tl == c_first));
        if (ok && a.emulate_slice && cnt != 0) {
          // the first staged span came from the chunk's first candidate with its start taken
          // at face value; the reference finds it by the reverse DFA over text[tp..]
          ulonglong2* sp = reinterpret_cast<ulonglong2*>(a.stage) + k * (uint64_t)a.stage_cap;
          const ulonglong2 first = sp[0];
          const uint64_t ms = slice_start(a.rev, a.text, a.n, tp, first.y, tp == a.clamp_p ? a.floor_flag : nullptr);
          if (ms == kNone || (ms == first.y) != (first.x == first.y) || cnt > a.stage_cap) ok = false;
          else if (ms != first.x) { sp[0].x = ms; a.meta[k] = meta | kMetaPatched; }
        }
        rewalk = !ok;
      } else if (tp > a.first_cand[k]) {
        if (!trim_staged(a, k, tp, cnt, &new_skip)) rewalk = true;
        else new_count = cnt - new_skip;
      }
    } else {
      // (a deferred chunk walked from its exact entry is waiting for the host to measure a long run)
      rewalk = state == kChunkDeferred || a.in_p[k] != tp || (strict && a.in_lm[k] != tl);
    }
    if (rewalk) {
      a.in_p[k] = tp;
      a.in_lm[k] = tl;
      a.dirty_list[atomicAdd(&counters[0], 1u)] = (uint32_t)k;
      atomicMin(&counters[3], (uint32_t)k);
      continue;
    }
    if (state != new_state || a.skip[k] != new_skip || a.count[k] != new_count) {
      a.meta[k] = (a.meta[k] & (kMetaCount | kMetaPatched)) | (new_state << 30);
      a.skip[k] = new_skip;
      a.count[k] = new_count;
      atomicAdd(&counters[1], 1u);
    }
  }
}

// Last resort for chains that never meet again (e.g. `(?s).{7}` tiling the haystack out of
// phase with every chunk): ONE thread walks chunk after chunk from a.seq_from to the end, each
// entered with its predecessor's exact exit state.  Linear time, no host round trips; the
// stitch loop then finds everything at and after seq_from consistent.
template <int FAST>
__global__ void __launch_bounds__(256) walk_sequential(WalkArgs a) {
  const auto R = RunnerSetup<FAST>::make(a);
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  Chain c;
  c.p = a.in_p[a.seq_from];
  c.lm = a.in_lm[a.seq_from];
  c.chain = c.p != kSpec;
  for (uint64_t k = a.seq_from; k < a.n_chunks; k++) {
    const bool spec = !c.chain;  // only the first chunk of a speculatively entered shard
    if (spec) { c.p = a.base + k * (uint64_t)a.chunk + 1; c.lm = kNone; }
    else { a.in_p[k] = c.p; a.in_lm[k] = c.lm; }
    uint64_t fc = kNone, total = 0;
    if (c.p != kNone) total = chunk_walk(a, R, k, c, &fc, a.stage, k * (uint64_t)a.stage_cap, (k + 1) * (uint64_t)a.stage_cap);
    finish_chunk(a, k, c, total, fc, spec);
    if (fc == kTooLong) return;  // a long run went to the host: the stitch loop resumes from this chunk once it is measured
    c.chain = true;  // an IDENT first chunk hands on its assumed first position: nothing lies before it in this shard
  }
}
template __global__ void walk_sequential<0>(WalkArgs);
template __global__ void walk_sequential<1>(WalkArgs);
template __global__ void walk_sequential<2>(WalkArgs);

// ------------------------------------------------------------- prefix sums ----
__device__ __forceinline__ uint64_t block_exclusive_scan(uint64_t v, uint64_t* total, uint64_t* warp_sums) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint64_t x = v;
  for (int o = 1; o < 32; o <<= 1) {
    uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_sums[wid] = x;
  __syncthreads();
  if (wid == 0) {
    uint64_t ws = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      uint64_t y = __shfl_up_sync(0xffffffffu, ws, o);
      if (lane >= o) ws += y;
    }
    warp_sums[lane] = ws;  // inclusive
  }
  __syncthreads();
  uint64_t warp_off = wid ? warp_sums[wid - 1] : 0;
  *total = warp_sums[(blockDim.x >> 5) - 1];
  return warp_off + x - v;
}
__global__ void scan_counts_local(const uint64_t* in, uint64_t* out, uint64_t* block_sums, uint64_t n) {
  __shared__ uint64_t ws[32];
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  uint64_t v = i < n ? in[i] : 0, total;
  uint64_t ex = block_exclusive_scan(v, &total, ws);
  if (i < n) out[i] = ex;
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}
__global__ void scan_block_sums(uint64_t* block_sums, uint64_t n_blocks, unsigned long long* grand_total) {
  __shared__ uint64_t ws[32];
  __shared__ uint64_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (uint64_t base = 0; base < n_blocks; base += blockDim.x) {
    uint64_t i = base + threadIdx.x;
    uint64_t v = i < n_blocks ? block_sums[i] : 0, total;
    uint64_t ex = block_exclusive_scan(v, &total, ws);
    uint64_t carry = carry_s;
    if (i < n_blocks) block_sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *grand_total = carry_s;
}
__global__ void scan_add_block_offsets(uint64_t* out, const uint64_t* block_sums, uint64_t n) {
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] += block_sums[blockIdx.x];
}

// ------------------------------------------------- replace_all / split ----------
// Bulk forms of the reference's thin loops over find_iter (src/re_bytes.rs:476-535 replacen,
// :316-360 / :699-749 split): the spans are on the device already, so the haystack never
// leaves it.
__global__ void span_lengths(const uint64_t* spans, uint64_t n_matches, uint64_t* lens) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_matches; i += (uint64_t)gridDim.x * blockDim.x)
    lens[i] = spans[2 * i + 1] - spans[2 * i];
}
__global__ void add_to_words(uint64_t* words, uint64_t n, uint64_t add) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) words[i] += add;
}
// span of group g of match i (kNone start = the group did not take part: expands to nothing)
__device__ __forceinline__ void rep_group(const ReplaceArgs& a, uint64_t i, uint32_t g, uint64_t* s, uint64_t* e) {
  if (g == 0 || !a.slots) { *s = a.spans[2 * i]; *e = a.spans[2 * i + 1]; return; }
  *s = a.slots[i * a.n_slots + 2 * g];
  *e = a.slots[i * a.n_slots + 2 * g + 1];
  if (*s == kNone || *e == kNone) *s = *e = 0;
}
__global__ void replace_lengths(ReplaceArgs a, uint64_t* rep_lens) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < a.n_matches; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t len = a.lit_total;
    for (uint32_t p = 0; p < a.n_parts; p++)
      if (a.part_len[p] & kRepGroup) {
        uint64_t s, e;
        rep_group(a, i, a.part_len[p] & ~kRepGroup, &s, &e);
        len += e - s;
      }
    rep_lens[i] = len;
  }
}
// The unmatched text.  One warp per 2 KiB tile of the INPUT (balanced whatever the gap sizes):
// binary search for the first match that ends after the tile's first byte, then gap by gap.
// With P_i / R_i = total length of the matches / replacements before match i, input byte x in the
// gap in front of match i lands at x - P_i + R_i.
__global__ void replace_gaps(ReplaceArgs a, uint64_t matched_total, uint64_t replaced_total) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  const uint64_t tiles = (a.n + 2047) / 2048;
  for (uint64_t t = warp; t < tiles; t += n_warps) {
    const uint64_t lo = t * 2048, hi = min(lo + 2048, a.n);
    uint64_t i0 = 0, i1 = a.n_matches;  // first match with end > lo
    while (i0 < i1) {
      const uint64_t mid = (i0 + i1) >> 1;
      if (a.spans[2 * mid + 1] <= lo) i0 = mid + 1; else i1 = mid;
    }
    uint64_t x = lo;
    for (uint64_t i = i0; x < hi; i++) {
      const bool tail = i >= a.n_matches;
      const uint64_t ms = tail ? a.n : a.spans[2 * i], me = tail ? a.n : a.spans[2 * i + 1];
      const int64_t shift = tail ? (int64_t)replaced_total - (int64_t)matched_total : (int64_t)a.reps_before[i] - (int64_t)a.lens_before[i];
      const uint64_t ge = min(ms, hi);  // gap [x, ge)
      for (uint64_t q = x + lane; q < ge; q += 32) {
        const uint64_t o = (uint64_t)((int64_t)q + shift);
        if (o < a.out_cap) a.out[o] = a.text[q];
      }
      if (tail) break;
      x = max(x, me);
    }
  }
}
// The replacements.  One warp per match.
__global__ void replace_matches(ReplaceArgs a) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t i = warp; i < a.n_matches; i += n_warps) {
    uint64_t o = a.spans[2 * i] - a.lens_before[i] + a.reps_before[i];
    for (uint32_t p = 0; p < a.n_parts; p++) {
      uint64_t len;
      const uint8_t* src;
      if (a.part_len[p] & kRepGroup) {
        uint64_t s, e;
        rep_group(a, i, a.part_len[p] & ~kRepGroup, &s, &e);
        len = e - s;
        src = a.text + s;
      } else {
        len = a.part_len[p];
        src = a.lits + a.part_off[p];
      }
      for (uint64_t q = lane; q < len; q += 32)
        if (o + q < a.out_cap) a.out[o + q] = src[q];
      o += len;
    }
  }
}
// Split (re_bytes.rs:699-721): piece i is the text between match i-1 and match i; the text after
// the last match is a piece only when it is not empty; SplitN (:734-749): the n-th piece is the rest.
__device__ __forceinline__ void split_piece(const uint64_t* spans, uint64_t n_matches, uint64_t n, uint64_t n_pieces, int last_is_rest, uint64_t i,
                                            uint64_t* piece) {
  piece[0] = i == 0 ? 0 : (i - 1 < n_matches ? spans[2 * (i - 1) + 1] : n);
  piece[1] = (i < n_matches && !(last_is_rest && i + 1 == n_pieces)) ? spans[2 * i] : n;
}
__global__ void split_pieces(const uint64_t* spans, uint64_t n_matches, uint64_t n, uint64_t n_pieces, int last_is_rest, uint64_t* pieces, uint64_t cap) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_pieces && i < cap; i += (uint64_t)gridDim.x * blockDim.x)
    split_piece(spans, n_matches, n, n_pieces, last_is_rest, i, pieces + 2 * i);
}

// ------------------------------------ batched records: replacen / splitn / captures_iter ----
// Per-record forms of the loops above.  Every item (match, piece) finds its record by a binary search in a CSR
// list rather than one thread walking each record, so a record with a million matches does not serialise.
// The record of item i: the last r with csr[r] <= i (csr[0] = 0 <= i < csr[n_rec]; empty records are passed over).
__device__ __forceinline__ uint64_t csr_row(const uint64_t* csr, uint64_t n_rec, uint64_t i) {
  uint64_t lo = 0, hi = n_rec;
  while (hi - lo > 1) {
    const uint64_t mid = (lo + hi) >> 1;
    if (csr[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}
__global__ void csr_counts(const uint64_t* csr, uint64_t n_rec, uint64_t limit, uint64_t* counts) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r <= n_rec; r += (uint64_t)gridDim.x * blockDim.x)
    counts[r] = r < n_rec ? min(csr[r + 1] - csr[r], limit) : 0;
}
__global__ void batch_keep_spans(const uint64_t* csr, const uint64_t* kcsr, uint64_t n_rec, const uint64_t* spans, uint64_t m, uint64_t* kept) {
  for (uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; j < m; j += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = csr_row(csr, n_rec, j), i = j - csr[r];
    if (i < kcsr[r + 1] - kcsr[r]) {
      kept[2 * (kcsr[r] + i)] = spans[2 * j];
      kept[2 * (kcsr[r] + i) + 1] = spans[2 * j + 1];
    }
  }
}
__global__ void batch_to_base(const uint64_t* offsets, const uint64_t* csr, uint64_t n_rec, uint64_t* spans, uint64_t m, uint64_t* slots,
                              uint32_t n_slots) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t b = offsets[csr_row(csr, n_rec, i)] - offsets[0];
    spans[2 * i] += b;
    spans[2 * i + 1] += b;
    if (slots)
      for (uint32_t k = 0; k < n_slots; k++)
        if (slots[i * n_slots + k] != kNone) slots[i * n_slots + k] += b;
  }
}
// With the spans of all records in one ordered list relative to offsets[0], the records' outputs are the pieces of
// the concatenated output: record r's output begins where its first kept match K would have landed had it been
// its first byte, i.e. at (offsets[r] - offsets[0]) - L[K] + P[K] (replace_gaps' shift).
__global__ void batch_replace_offsets(const uint64_t* offsets, const uint64_t* csr, uint64_t n_rec, const uint64_t* lens_before,
                                      const uint64_t* reps_before, uint64_t m, uint64_t matched_total, uint64_t replaced_total,
                                      uint64_t* out_offsets) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r <= n_rec; r += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t k = csr[r];
    const uint64_t l = k < m ? lens_before[k] : matched_total, p = k < m ? reps_before[k] : replaced_total;
    out_offsets[r] = offsets[r] - offsets[0] - l + p;
  }
}
// split_device per record: one piece per match, the rest when it is not empty; SplitN clamps to `limit`, and the
// limit-th piece is the rest (so limit 0 gives none and limit 1 the whole record, even an empty one)
__global__ void batch_split_counts(const uint64_t* offsets, const uint64_t* csr, const uint64_t* spans, uint64_t n_rec, int has_limit,
                                   uint64_t limit, uint64_t* counts) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r <= n_rec; r += (uint64_t)gridDim.x * blockDim.x) {
    if (r == n_rec) { counts[r] = 0; continue; }
    const uint64_t c = csr[r + 1] - csr[r], len = offsets[r + 1] - offsets[r];
    const uint64_t last_end = c ? spans[2 * (csr[r + 1] - 1) + 1] : 0;
    uint64_t p = c + (last_end < len ? 1 : 0);
    if (has_limit && p + 1 >= limit) p = limit;
    counts[r] = p;
  }
}
__global__ void batch_split_pieces(const uint64_t* offsets, const uint64_t* csr, const uint64_t* spans, const uint64_t* pcsr, uint64_t n_rec,
                                   int has_limit, uint64_t limit, uint64_t* pieces, uint64_t n_out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_out; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = csr_row(pcsr, n_rec, i), np = pcsr[r + 1] - pcsr[r];
    // a record has `limit` pieces only when the SplitN clamp applied (otherwise it has fewer than limit - 1)
    split_piece(spans + 2 * csr[r], csr[r + 1] - csr[r], offsets[r + 1] - offsets[r], np, has_limit && np == limit, i - pcsr[r], pieces + 2 * i);
  }
}
__global__ void batch_diverged(const uint64_t* csr, uint64_t n_rec, const uint64_t* spans, uint64_t m, const uint64_t* slots, uint32_t n_slots,
                               uint32_t* flags, uint64_t* list, unsigned int* n_list) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  uint64_t r = 0;
  bool first = false;
  if (i < m && (slots[i * n_slots] != spans[2 * i] || slots[i * n_slots + 1] != spans[2 * i + 1])) {
    r = csr_row(csr, n_rec, i);
    const uint32_t bit = 1u << (r & 31);
    first = !(atomicOr(&flags[r >> 5], bit) & bit);
  }
  const uint32_t b = __ballot_sync(0xffffffffu, first);
  if (!b) return;
  const int leader = __ffs(b) - 1;
  unsigned int base = 0;
  if ((int)lane == leader) base = atomicAdd(n_list, (unsigned int)__popc(b));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (first) list[base + __popc(b & ((1u << lane) - 1))] = r;
}
__global__ void batch_move_rows(const uint64_t* csr, const uint64_t* new_csr, uint64_t n_rec, const uint32_t* skip, const uint64_t* src, uint64_t m,
                                uint32_t width, uint64_t* dst, uint64_t cap) {
  for (uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; j < m; j += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = csr_row(csr, n_rec, j);
    if ((skip[r >> 5] >> (r & 31)) & 1u) continue;
    const uint64_t d = new_csr[r] + (j - csr[r]);
    if (d >= cap) continue;
    for (uint32_t k = 0; k < width; k++) dst[d * width + k] = src[j * width + k];
  }
}

// ----------------------------------------------------------- capture groups ----
// The reference fills `Captures` by running its NFA simulation over the window the DFA
// narrowed down: from the match start to two characters past the match end
// (src/exec.rs:861-875 captures_nfa_with_match).  Same here: one thread per match runs the Pike
// VM of src/pikevm.rs:130-352 (thread lists in priority order, per-thread slot arrays, the
// explicit stack that restores slots behind a Save) over the capture program -- the forward
// program, lazy prefix included, compiled WITH Save instructions.  (The search starts at the
// match start the DFA found; where the reverse-on-slice quirk of SURVEY H1 made that start one
// no match begins at, the NFA reports the next match inside the window or none, as it does in
// the reference.)  Scratch lives in global memory, one slab per
// resident thread; this is a per-match O(window x program) pass, not a streaming kernel.
__device__ __forceinline__ bool look_holds(uint32_t look, const uint8_t* t, uint64_t n, uint64_t at) {  // src/input.rs:268-318
  const bool w1 = at > 0 && is_word_byte(t[at - 1]);
  const bool w2 = at < n && is_word_byte(t[at]);
  switch (look) {
    case 0: return at == 0 || t[at - 1] == '\n';  // StartLine
    case 1: return at == n || t[at] == '\n';      // EndLine
    case 2: return at == 0;                        // StartText
    case 3: return at == n;                        // EndText
    case 4: case 6: return w1 != w2;               // word boundary (ASCII; the Unicode one is rejected at compile time)
    default: return w1 == w2;
  }
}
struct PikeList {
  uint32_t* sparse;
  uint32_t* dense;
  uint64_t* caps;  // [ip][slot]
  uint32_t count;
  __device__ __forceinline__ bool contains(uint32_t ip) const { const uint32_t i = sparse[ip]; return i < count && dense[i] == ip; }
  __device__ __forceinline__ void insert(uint32_t ip) { sparse[ip] = count; dense[count++] = ip; }
};
// pikevm.rs:274-352: follow the epsilon transitions from ip0 in priority order
__device__ void pike_add(const CapArgs& a, const uint8_t* text, PikeList& l, uint64_t* tc, uint32_t ip0, uint64_t n, uint64_t at, uint32_t* stk_tag, uint64_t* stk_pos) {
  uint32_t sp = 0;
  stk_tag[sp] = ip0; stk_pos[sp++] = 0;  // tag < 0x80000000: an instruction to visit; else: restore slot (tag & 0x7FFFFFFF) to pos
  while (sp) {
    --sp;
    const uint32_t tag = stk_tag[sp];
    if (tag & 0x80000000u) { tc[tag & 0x7FFFFFFFu] = stk_pos[sp]; continue; }
    uint32_t ip = tag;
    for (;;) {
      if (l.contains(ip)) break;
      l.insert(ip);
      const NfaInst in = a.insts[ip];
      const uint32_t op = in.op_look_lo_hi & 0xFF;
      if (op == 3) {         // EmptyLook
        if (!look_holds((in.op_look_lo_hi >> 8) & 0xFF, text, n, at)) break;
        ip = in.a;
      } else if (op == 1) {  // Save
        if (in.b < a.n_slots) {
          stk_tag[sp] = 0x80000000u | in.b; stk_pos[sp++] = tc[in.b];
          tc[in.b] = at;
        }
        ip = in.a;
      } else if (op == 2) {  // Split: goto1 first, goto2 later
        stk_tag[sp] = in.b; stk_pos[sp++] = 0;
        ip = in.a;
      } else {               // Match or Bytes: the thread waits here with its slots
        for (uint32_t k = 0; k < a.n_slots; k++) l.caps[(uint64_t)ip * a.n_slots + k] = tc[k];
        break;
      }
    }
  }
}
__global__ void pike_captures(CapArgs a) {
  const uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint64_t n_threads = (uint64_t)gridDim.x * blockDim.x;
  uint8_t* mine = a.scratch + tid * a.per_thread;
  const uint64_t ni = a.n_insts, ns = a.n_slots;
  PikeList L[2];
  uint64_t off = 0;
  for (int j = 0; j < 2; j++) { L[j].caps = reinterpret_cast<uint64_t*>(mine + off); off += ni * ns * 8; }
  uint64_t* tc = reinterpret_cast<uint64_t*>(mine + off); off += ns * 8;
  uint64_t* stk_pos = reinterpret_cast<uint64_t*>(mine + off); off += (2 * ni + 4) * 8;
  for (int j = 0; j < 2; j++) { L[j].sparse = reinterpret_cast<uint32_t*>(mine + off); off += ni * 4; L[j].dense = reinterpret_cast<uint32_t*>(mine + off); off += ni * 4; }
  uint32_t* stk_tag = reinterpret_cast<uint32_t*>(mine + off);
  for (uint64_t m = tid; m < a.n_matches; m += n_threads) {
    const uint64_t s = a.spans[2 * m], e = a.spans[2 * m + 1];
    uint64_t* out = a.slots + m * ns;
    for (uint32_t k = 0; k < ns; k++) { out[k] = kNone; tc[k] = kNone; }
    const uint8_t* text = a.text;  // the text the match is relative to: the haystack, or record m
    uint64_t tn = a.n;
    if (a.rec_offsets) {
      uint64_t r = m;
      if (a.rec_csr) r = csr_row(a.rec_csr, a.n_rec, m);
      else if (!((a.rec_found[m >> 5] >> (m & 31)) & 1u)) continue;
      text = a.text + a.rec_offsets[r];
      tn = a.rec_offsets[r + 1] - a.rec_offsets[r];
    }
    // the window ends two characters past the match (look-ahead needs them; utf8.rs:24-40 next_utf8)
    uint64_t n = e;
    for (int r = 0; r < 2; r++) {
      if (n >= tn) { n = tn; break; }
      const uint32_t b = text[n];
      n += b <= 0x7F ? 1 : b <= 0xDF ? 2 : b <= 0xEF ? 3 : 4;
    }
    n = min(n, tn);
    int cur = 0;
    L[0].count = L[1].count = 0;
    for (uint64_t i = 0; i < ni; i++) L[0].sparse[i] = L[1].sparse[i] = 0;
    bool matched = false;
    for (uint64_t at = s;; at++) {
      PikeList& cl = L[cur];
      PikeList& nl = L[cur ^ 1];
      if (cl.count == 0 && (matched || (at != 0 && a.anchored_start))) break;  // pikevm.rs:143-158
      // a new thread at every position until something has matched: the program's lazy prefix
      // (pikevm.rs:172-175); its slots start out empty
      if (cl.count == 0 || (!a.anchored_start && !matched)) {
        for (uint32_t k = 0; k < ns; k++) tc[k] = kNone;
        pike_add(a, text, cl, tc, a.start_ip, n, at, stk_tag, stk_pos);
      }
      for (uint32_t i = 0; i < cl.count; i++) {
        const uint32_t ip = cl.dense[i];
        const NfaInst in = a.insts[ip];
        const uint32_t op = in.op_look_lo_hi & 0xFF;
        if (op == 0) {  // Match: leftmost-first -- lower-priority threads of this step are dropped
          for (uint32_t k = 0; k < ns; k++) out[k] = cl.caps[(uint64_t)ip * ns + k];
          matched = true;
          break;
        }
        if (op == 4 && at < n) {  // Bytes
          const uint32_t b = text[at];
          if (((in.op_look_lo_hi >> 16) & 0xFF) <= b && b <= (in.op_look_lo_hi >> 24)) {
            for (uint32_t k = 0; k < ns; k++) tc[k] = cl.caps[(uint64_t)ip * ns + k];
            pike_add(a, text, nl, tc, in.a, n, at + 1, stk_tag, stk_pos);
          }
        }
      }
      if (at >= n) break;
      cl.count = 0;
      cur ^= 1;
    }
  }
}

__global__ void slot_found_bits(const uint64_t* slots, uint32_t n_slots, uint64_t n_rec, uint32_t* bits) {
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint32_t b = __ballot_sync(0xffffffffu, r < n_rec && slots[r * n_slots] != kNone);
  if ((threadIdx.x & 31) == 0 && r < n_rec) bits[r >> 5] = b;
}

// ---------------------------------------------------------------- batch mode --
// One thread per record; each record is its own haystack (record-local ^, $, \b).
__global__ void is_match_batch(BatchArgs a) {
  const Table T = stage_table(a.fwd, g_smem, a.use_smem);
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  bool matched = false;
  if (r < a.n_rec) {
    const uint64_t lo = a.offsets[r], len = a.offsets[r + 1] - lo;
    matched = earliest_end(a.fwd, T, a.text + lo, len, 0) != kNone;
  }
  const uint32_t bits = __ballot_sync(0xffffffffu, matched);
  if ((threadIdx.x & 31) == 0 && r < a.n_rec) a.out_bits[r >> 5] = bits;
}

// exec.rs:632-662 per record on the class-indexed tables in global memory: forward leftmost-first end e, then
// the start ms by the reverse longest automaton over the record.  false: no match (ms, me left as they are).
// The forward loop is anchored_end's with plain loads instead of __ldg: through slow_find_record, __ldg here
// changes the code of batch_fast<1> and costs it 0.4 % on C3 find (B200, 1000 W).
__device__ __forceinline__ bool find_in_record(const DfaView& f, const DfaView& rv, const uint8_t* p, uint64_t len, uint64_t& ms,
                                               uint64_t& me) {
  uint32_t st = pick_start_fwd(f, p, len, 0);
  uint64_t e = kNone;
  for (uint64_t q = 0; st != 0; q++) {
    st = q < len ? f.trans[st * f.stride + f.classes[p[q]]] : f.trans[st * f.stride + f.stride - 1];
    if (st >= f.match_lo) e = q;
    if (q >= len) break;
  }
  if (e == kNone) return false;
  const uint64_t s = e == 0 ? 0 : slice_start(rv, p, len, 0, e);
  if (s == kNone) return false;
  ms = s;
  me = e;
  return true;
}

__global__ void find_batch(BatchArgs a) {
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  bool found = false;
  if (r < a.n_rec) {
    const uint64_t lo = a.offsets[r], len = a.offsets[r + 1] - lo;
    uint64_t ms, me;
    if (find_in_record(a.fwd, a.rev, a.text + lo, len, ms, me)) {
      found = true;
      a.out_spans[2 * r] = ms;
      a.out_spans[2 * r + 1] = me;
    } else {
      a.out_spans[2 * r] = 0;
      a.out_spans[2 * r + 1] = 0;
    }
  }
  const uint32_t bits = __ballot_sync(0xffffffffu, found);
  if ((threadIdx.x & 31) == 0 && r < a.n_rec) a.out_bits[r >> 5] = bits;
}


// ---- batch_fast: the same per-record algorithms on the shared-memory hot tables ----
// One thread per record as above, but (a) one LDS per byte on the byte-indexed tables
// instead of class + transition look-ups, (b) the record is read 16 bytes at a time from
// three aligned 8-byte loads (a byte load per lane costs a full L1 wavefront per lane:
// 32 per warp-step, against ~2 for the table), (c) persistent blocks, so the tables are
// staged once per block.  A record that leaves the hot set is redone on the full tables.
__device__ __forceinline__ void window16(const uint8_t* p, uint32_t (&v)[4]) {
  const uintptr_t addr = reinterpret_cast<uintptr_t>(p);
  const uint64_t* wp = reinterpret_cast<const uint64_t*>(addr & ~(uintptr_t)7);
  const uint32_t sh = (uint32_t)(addr & 7) * 8;
  const uint64_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
  const uint32_t x0 = __funnelshift_r((uint32_t)w0, (uint32_t)(w0 >> 32), sh);
  const uint32_t x1 = __funnelshift_r((uint32_t)(w0 >> 32), (uint32_t)w1, sh);
  const uint32_t x2 = __funnelshift_r((uint32_t)w1, (uint32_t)(w1 >> 32), sh);
  const uint32_t x3 = __funnelshift_r((uint32_t)(w1 >> 32), (uint32_t)w2, sh);
  const uint32_t x4 = __funnelshift_r((uint32_t)w2, (uint32_t)(w2 >> 32), sh);
  const bool up = sh >= 32;
  v[0] = up ? x1 : x0; v[1] = up ? x2 : x1; v[2] = up ? x3 : x2; v[3] = up ? x4 : x3;
}
// The same window from two aligned 16-byte loads (reads [p & ~15, (p & ~15) + 32)): two L1 wavefronts per
// lane instead of three -- the batch kernels are bound by exactly those (every lane reads its own line).
__device__ __forceinline__ void window16q(const uint8_t* p, uint32_t (&v)[4]) {
  const uintptr_t addr = reinterpret_cast<uintptr_t>(p);
  const uint8_t* al = reinterpret_cast<const uint8_t*>(addr & ~(uintptr_t)15);
  const uint4 p0 = ldg128(al), p1 = ldg128(al + 16);
  const bool by2 = (addr & 8u) != 0, by1 = (addr & 4u) != 0;
  const uint32_t sh = (uint32_t)(addr & 3u) * 8u;
  const uint32_t a0 = by2 ? p0.z : p0.x, a1 = by2 ? p0.w : p0.y, a2 = by2 ? p1.x : p0.z, a3 = by2 ? p1.y : p0.w,
                 a4 = by2 ? p1.z : p1.x, a5 = by2 ? p1.w : p1.y;
  const uint32_t b0 = by1 ? a1 : a0, b1 = by1 ? a2 : a1, b2 = by1 ? a3 : a2, b3 = by1 ? a4 : a3, b4 = by1 ? a5 : a4;
  v[0] = __funnelshift_r(b0, b1, sh); v[1] = __funnelshift_r(b1, b2, sh);
  v[2] = __funnelshift_r(b2, b3, sh); v[3] = __funnelshift_r(b3, b4, sh);
}
__device__ __forceinline__ uint32_t window_byte(const uint32_t (&v)[4], int i) {  // byte i, i compile-time
  return (v[i >> 2] >> (8 * (i & 3))) & 0xFFu;
}
// A record that left the hot set, again on the full tables (pointer arguments for the reason given at
// slow_anchored_end).
__device__ __noinline__ bool slow_is_match_record(const DfaView* f, const uint8_t* p, uint64_t len) {
  return earliest_end(*f, global_table(*f), p, len, 0) != kNone;
}
__device__ __noinline__ bool slow_find_record(const DfaView* f, const DfaView* rv, const uint8_t* p, uint64_t len, uint64_t* ms_out, uint64_t* e_out) {
  return find_in_record(*f, *rv, p, len, *ms_out, *e_out);
}

// The forward loop of batch_fast: record bytes from q on, hot state e on entry (the start state for
// position q), 16 bytes per window.  MODE 0: stops at the first match state, mx = highest state seen;
// MODE 1: runs until the automaton dies, last = end of the leftmost-first match (kNone: none).
// On return e == 1 (trap) means the record left the hot set: redo it on the full tables.
template <int MODE>
__device__ __forceinline__ void hot_forward(const BatchArgs& a, uint32_t fbase, const uint8_t* p, uint64_t len, uint64_t q,
                                            const uint8_t* buf_hi, uint32_t& e, uint64_t& last, uint32_t& mx) {
  const uint32_t fthr = a.fwd_hot.match_lo, flive = 2;
  bool done = false;
  while (!done) {
    const uint64_t left = len - q;
    if (left == 0) {  // EOF step
      if (e >= flive && a.fwd_hot.eof[e] >= a.fwd.match_lo) { last = len; mx = 0xFFFFFFFFu; }
      break;
    }
    const uint8_t* wp = p + q;
    const uint8_t* al = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(wp) & ~(uintptr_t)7);
    if (al + 24 <= buf_hi) {
      uint32_t v[4];
      window16(wp, v);
      const uint32_t nb = left >= 16 ? 16u : (uint32_t)left;
      uint32_t lj = ~0u;
      if (nb == 16) {
#pragma unroll
        for (int g = 0; g < 4; g++) {
          e = hot_next<0>(fbase, v[g], e); if (MODE == 0) mx = max(mx, e); else if (e >= fthr) lj = 4 * g + 0;
          e = hot_next<1>(fbase, v[g], e); if (MODE == 0) mx = max(mx, e); else if (e >= fthr) lj = 4 * g + 1;
          e = hot_next<2>(fbase, v[g], e); if (MODE == 0) mx = max(mx, e); else if (e >= fthr) lj = 4 * g + 2;
          e = hot_next<3>(fbase, v[g], e); if (MODE == 0) mx = max(mx, e); else if (e >= fthr) lj = 4 * g + 3;
          if (e < flive || (MODE == 0 && mx >= fthr)) { done = true; break; }
        }
      } else {
#pragma unroll
        for (int i = 0; i < 15; i++) {
          if ((uint32_t)i < nb) {
            e = hot_next_b(fbase, window_byte(v, i), e);
            if (MODE == 0) mx = max(mx, e);
            else if (e >= fthr) lj = i;
          }
        }
        if (e < flive || (MODE == 0 && mx >= fthr)) done = true;
      }
      if (MODE == 1 && lj != ~0u) last = q + lj;
      q += nb;
    } else {  // the last bytes of the whole buffer: byte loads
      for (uint64_t i = 0; i < left && !done; i++) {
        e = hot_next_b(fbase, p[q + i], e);
        if (MODE == 0) mx = max(mx, e);
        else if (e >= fthr) last = q + i;
        if (e < flive || (MODE == 0 && mx >= fthr)) done = true;
      }
      q += left;
    }
  }
}

// The reverse loop of batch_fast: start of the match that ends at me > lo, found by the reverse longest
// automaton over the slice p[lo..] (exec.rs:651-657; lo is that slice's beginning of text).  kNone: no
// start.  rcold: the scan left the hot set and must be redone on the full tables (slice_start).
__device__ __forceinline__ uint64_t hot_reverse(const BatchArgs& a, uint32_t rbase, const uint8_t* p, uint64_t len, uint64_t lo,
                                                uint64_t me, const uint8_t* buf_hi, bool& rcold) {
  const uint32_t rthr = a.rev_hot.match_lo, rlive = 2;
  uint64_t start = kNone;
  // flags at me of the slice p[lo..] are those of the record: me > lo
  const uint32_t sf = a.rev.uniform_start ? a.rev.start[32] : a.rev.start[flags_reverse(p, len, me)];
  const uint32_t hr = a.rev_hot.full2hot[sf];
  if (sf == 0) {
    start = kNone;
  } else if (hr == 0xFFFFu) {
    rcold = true;
  } else {
    uint32_t er = hr;
    uint64_t at = me;
    bool rdone = false;
    while (at > lo && !rdone) {
      const uint8_t* wp = p + at - 16;  // window = bytes [at-16, at); only the last min(16, at - lo) belong to the slice
      const uint8_t* al = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(wp) & ~(uintptr_t)7);
      const uint32_t nb = at - lo >= 16 ? 16u : (uint32_t)(at - lo);
      if (al >= a.text && al + 24 <= buf_hi) {
        uint32_t v[4];
        window16(wp, v);
        uint32_t lj = ~0u;
#pragma unroll
        for (int i = 15; i >= 0; i--) {
          if ((uint32_t)(15 - i) < nb && !rdone) {
            er = hot_next_b(rbase, window_byte(v, i), er);
            if (er >= rthr) lj = i;
            if (er < rlive) rdone = true;
          }
        }
        if (lj != ~0u) start = at - 16 + lj + 1;
        at -= nb;
      } else {
        for (uint32_t i = 0; i < nb && !rdone; i++) {
          at--;
          er = hot_next_b(rbase, p[at], er);
          if (er >= rthr) start = at + 1;
          if (er < rlive) rdone = true;
        }
      }
    }
    if (er == 1u) rcold = true;
    else if (!rdone && a.rev_hot.eof[er] >= a.rev.match_lo) start = lo;
  }
  return start;
}

// MODE 0: is_match (forward all-match automaton, stop at the first match state);
// MODE 1: find (forward leftmost-first end, then the reverse longest automaton for the start).
template <int MODE>
__global__ void __launch_bounds__(512) batch_fast(BatchArgs a) {
  const uint32_t fbase = ((uint32_t)__cvta_generic_to_shared(g_smem) + 255u) & ~255u;
  const uint32_t rbase = fbase + hot_table_bytes(a.fwd_hot.n);
  hot_stage(a.fwd_hot, fbase);
  if (MODE == 1) hot_stage(a.rev_hot, rbase);
  __syncthreads();
  const uint32_t fthr = a.fwd_hot.match_lo;
  const uint8_t* const buf_hi = a.text + a.offsets[a.n_rec];
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;  // multiple of 32: warps stay on one ballot word
  const uint32_t lane = threadIdx.x & 31;
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r - lane < a.n_rec; r += stride) {
    bool hit = false;
    uint64_t ms = 0, me = 0;
    if (r < a.n_rec) {
      const uint64_t lo = a.offsets[r], len = a.offsets[r + 1] - lo;
      const uint8_t* p = a.text + lo;
      bool cold = false;
      // ---- forward ----
      const uint32_t h0 = a.fwd.uniform_start ? a.fwd_hot.start : a.fwd_hot.full2hot[a.fwd.start[flags_forward(p, len, 0)]];
      uint32_t e = h0 == 0xFFFFu ? 1u : h0;
      uint64_t last = kNone;
      uint32_t mx = 0;
      hot_forward<MODE>(a, fbase, p, len, 0, buf_hi, e, last, mx);
      if (e == 1u && !(MODE == 0 && mx >= fthr)) cold = true;  // trap row
      if (MODE == 0) {
        hit = cold ? slow_is_match_record(a.fwd_g, p, len) : mx >= fthr;
      } else if (cold) {
        hit = slow_find_record(a.fwd_g, a.rev_g, p, len, &ms, &me);
      } else if (last != kNone) {
        // ---- reverse from the match end (exec.rs:651-657; the record is its own slice) ----
        me = last;
        bool rcold = false;
        const uint64_t start = me == 0 ? 0 : hot_reverse(a, rbase, p, len, 0, me, buf_hi, rcold);
        if (rcold) {
          hit = slow_find_record(a.fwd_g, a.rev_g, p, len, &ms, &me);
        } else if (start != kNone) {
          hit = true;
          ms = start;
        }
      }
      if (MODE == 1) {
        a.out_spans[2 * r] = hit ? ms : 0;
        a.out_spans[2 * r + 1] = hit ? me : 0;
      }
    }
    const uint32_t bits = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) a.out_bits[r >> 5] = bits;
  }
}
template __global__ void batch_fast<0>(BatchArgs);
template __global__ void batch_fast<1>(BatchArgs);

// ---- batch_iter: find_iter per record (re_trait.rs:197-220 with the record as the whole text) ----
// From p: the end e of the leftmost-first match found from p (forward unanchored automaton, start state by
// the flags at p), its start by the reverse scan over the slice [p..] (exec.rs:651-657, so p is judged as
// beginning of text: SURVEY H1), then the empty-match rule (exec.rs:335-377).  Two launches of one kernel
// build the CSR output: PASS 0 counts the matches of each record, an exclusive scan turns the counts into
// offsets, PASS 1 runs the iterator again and stores.  Match counts per record are unbounded, so a single
// pass would need per-record staging of unbounded size; the second pass costs a second read of the text.
// fwd(q) -> match end or kNone; rev(q, e) -> match start (e > q) or kNone.
template <int PASS, class Fwd, class Rev>
__device__ __forceinline__ void iter_record(const BatchArgs& a, uint64_t r, const uint8_t* p, uint64_t len, Fwd fwd, Rev rev) {
  const uint64_t base = PASS == 1 ? a.match_offsets[r] : 0;
  uint64_t k = 0, q = 0, lm = kNone;
  while (q <= len) {
    const uint64_t e = fwd(q);
    if (e == kNone) break;
    if (PASS == 0 && a.fwd_only) {  // no empty match, no look-around: s < e and the reverse scan cannot fail
      k++;
      q = e;
      continue;
    }
    const uint64_t s = e == q ? q : rev(q, e);
    if (s == kNone) break;  // the reverse-on-slice scan failed: the reference's iteration ends here
    if (s == e) {
      q = a.utf8 ? next_utf8(p, len, e) : e + 1;
      if (e == lm) continue;
    } else {
      q = e;
    }
    lm = e;
    if (PASS == 1 && base + k < a.cap) {
      a.out_spans[2 * (base + k)] = s;
      a.out_spans[2 * (base + k) + 1] = e;
    }
    k++;
  }
  if (PASS == 0) a.match_offsets[r] = k;
}

// One thread per record on the hot tables, as batch_fast<1> (persistent blocks, 16-byte windows).  A
// record that leaves the hot set finishes its iteration on the full tables in global memory.
template <int PASS>
__global__ void __launch_bounds__(512, 2) batch_iter_fast(BatchArgs a) {
  const uint32_t fbase = ((uint32_t)__cvta_generic_to_shared(g_smem) + 255u) & ~255u;
  const uint32_t rbase = fbase + hot_table_bytes(a.fwd_hot.n);
  hot_stage(a.fwd_hot, fbase);
  hot_stage(a.rev_hot, rbase);
  __syncthreads();
  const uint8_t* const buf_hi = a.text + a.offsets[a.n_rec];
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < a.n_rec; r += stride) {
    const uint64_t lo = a.offsets[r], len = a.offsets[r + 1] - lo;
    const uint8_t* p = a.text + lo;
    bool cold = false;
    auto fwd = [&](uint64_t q) -> uint64_t {
      if (!cold) {
        const uint32_t h0 = a.fwd.uniform_start ? a.fwd_hot.start : a.fwd_hot.full2hot[a.fwd.start[flags_forward(p, len, q)]];
        uint32_t e = h0 == 0xFFFFu ? 1u : h0, mx = 0;
        uint64_t last = kNone;
        hot_forward<1>(a, fbase, p, len, q, buf_hi, e, last, mx);
        if (e != 1u) return last;
        cold = true;
      }
      return anchored_end(*a.fwd_g, global_table(*a.fwd_g), p, len, q);
    };
    auto rev = [&](uint64_t q, uint64_t e) -> uint64_t {
      if (!cold) {
        const uint64_t s = hot_reverse(a, rbase, p, len, q, e, buf_hi, cold);
        if (!cold) return s;
      }
      return slice_start(*a.rev_g, p, len, q, e);
    };
    iter_record<PASS>(a, r, p, len, fwd, rev);
  }
}
template __global__ void batch_iter_fast<0>(BatchArgs);
template __global__ void batch_iter_fast<1>(BatchArgs);

// Generic: one thread per record on the class-indexed tables (no hot set, unaligned haystacks, force_generic).
template <int PASS>
__global__ void batch_iter(BatchArgs a) {
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (r >= a.n_rec) return;
  const uint64_t lo = a.offsets[r], len = a.offsets[r + 1] - lo;
  const uint8_t* p = a.text + lo;
  iter_record<PASS>(a, r, p, len, [&](uint64_t q) { return anchored_end(a.fwd, global_table(a.fwd), p, len, q); },
                    [&](uint64_t q, uint64_t e) { return slice_start(a.rev, p, len, q, e); });
}
template __global__ void batch_iter<0>(BatchArgs);
template __global__ void batch_iter<1>(BatchArgs);

// ---- batch_refill: batch_fast<0> with the lanes of a warp kept busy ----
// batch_fast gives every lane one record and waits for the slowest of the 32: on log lines 70 % of the
// records are decided inside their first window and their lanes idle until the longest line of the warp
// is through (ncu: 8.5 of 32 threads per instruction).  Here a warp owns a task of kBatchTask consecutive
// records; a lane that has decided its record takes the next one of the task as soon as kBatchRefill lanes
// are free (the refill code runs for all of them together), so a step of the loop is one 16-byte window for
// (nearly) every lane.  Result bits are collected in shared memory and leave as whole words.
// is_match only: the same scheme for find (a forward loop, then a reverse loop for the starts) measured
// slower than batch_fast<1> on log lines (profiles/r02_ncu_summaries.md §3b).
constexpr uint32_t kBatchTask = 2048, kBatchRefill = 8;
__global__ void __launch_bounds__(512) batch_refill(BatchArgs a) {
  __shared__ uint32_t task_bits[16][kBatchTask / 32];  // blockDim.x == 512
  const uint32_t fbase = ((uint32_t)__cvta_generic_to_shared(g_smem) + 255u) & ~255u;
  hot_stage(a.fwd_hot, fbase);
  __syncthreads();
  const uint32_t fthr = a.fwd_hot.match_lo, flive = 2;
  const uint8_t* const buf_hi = a.text + a.offsets[a.n_rec];
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t task_recs = a.task_recs;  // multiple of 32, at most kBatchTask (the host sizes it so that every warp gets several)
  const uint64_t n_tasks = (a.n_rec + task_recs - 1) / task_recs;
  uint32_t* bits = task_bits[wid];
  for (;;) {
    // tasks are handed out through a global counter: with a fixed assignment the warps that get one task
    // more than the others decide the kernel's time
    unsigned long long task = 0;
    if (lane == 0) task = atomicAdd(a.task_counter, 1ull);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= n_tasks) break;
    const uint64_t r_lo = task * task_recs, r_hi = min(r_lo + task_recs, a.n_rec);
    for (uint32_t i = lane; i < task_recs / 32; i += 32) bits[i] = 0;
    __syncwarp();
    uint64_t next = r_lo;  // warp-uniform: first record of the task not handed out yet
    bool idle = true;
    uint64_t r = 0, len = 0, q = 0;
    const uint8_t* p = a.text;
    uint32_t e = 0, mx = 0;
    auto finish = [&](bool hit) {
      if (hit) atomicOr(&bits[(uint32_t)(r - r_lo) >> 5], 1u << ((uint32_t)(r - r_lo) & 31u));
      idle = true;
    };
    for (;;) {
      const uint32_t idle_m = __ballot_sync(0xffffffffu, idle);
      if (idle_m == 0xffffffffu && next >= r_hi) break;
      if (next < r_hi && ((uint32_t)__popc(idle_m) >= kBatchRefill || idle_m == 0xffffffffu)) {
        const uint64_t mine = next + (uint32_t)__popc(idle_m & ((1u << lane) - 1u));
        if (idle && mine < r_hi) {
          r = mine;
          const uint64_t lo = a.offsets[r];
          len = a.offsets[r + 1] - lo;
          p = a.text + lo;
          q = 0;
          mx = 0;
          const uint32_t h0 = a.fwd.uniform_start ? a.fwd_hot.start : a.fwd_hot.full2hot[a.fwd.start[flags_forward(p, len, 0)]];
          e = h0 == 0xFFFFu ? 1u : h0;
          idle = false;
        }
        next = min(next + (uint64_t)__popc(idle_m), r_hi);
      }
      if (idle) continue;
      bool done = false;
      const uint64_t left = len - q;
      if (left == 0) {  // EOF step
        if (e >= flive && a.fwd_hot.eof[e] >= a.fwd.match_lo) mx = 0xFFFFFFFFu;
        done = true;
      } else if (e < flive) {
        done = true;  // dead or trap from the start state
      } else {
        const uint8_t* wp = p + q;
        const uint8_t* al = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(wp) & ~(uintptr_t)15);
        if (al + 32 <= buf_hi) {
          uint32_t v[4];
          window16q(wp, v);
          const uint32_t nb = left >= 16 ? 16u : (uint32_t)left;
          if (nb == 16) {
#pragma unroll
            for (int g = 0; g < 4; g++) {
              e = hot_next<0>(fbase, v[g], e); mx = max(mx, e);
              e = hot_next<1>(fbase, v[g], e); mx = max(mx, e);
              e = hot_next<2>(fbase, v[g], e); mx = max(mx, e);
              e = hot_next<3>(fbase, v[g], e); mx = max(mx, e);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 15; i++)
              if ((uint32_t)i < nb) {
                e = hot_next_b(fbase, window_byte(v, i), e);
                mx = max(mx, e);
              }
          }
          q += nb;
        } else {  // the last bytes of the whole buffer: byte loads
          for (uint64_t i = 0; i < left && e >= flive && mx < fthr; i++) {
            e = hot_next_b(fbase, p[q + i], e);
            mx = max(mx, e);
          }
          q += left;
        }
        if (e < flive || mx >= fthr) done = true;
      }
      if (done) {
        if (e == 1u && !(mx >= fthr)) finish(slow_is_match_record(a.fwd_g, p, len));  // left the hot set: again on the full tables
        else finish(mx >= fthr);
      }
    }
    __syncwarp();
    for (uint32_t i = lane; i < task_recs / 32; i += 32)
      if (r_lo + 32ull * i < r_hi) a.out_bits[(r_lo >> 5) + i] = bits[i];
    __syncwarp();
  }
}

// dfa.rs:525-570 per record: OR of the per-state pattern masks of automaton d along the scan of record r.
__device__ __forceinline__ void set_record_masks(const Table& T, const DfaView& d, const uint8_t* text, const uint64_t* offsets,
                                                 uint64_t n_rec, uint64_t r, uint64_t (&acc)[kMaxMaskWords]) {
  const uint64_t lo = offsets[r], len = offsets[r + 1] - lo;
  const uint8_t* p = text + lo;
  const uint32_t mw = d.mask_words;
  uint32_t s = pick_start_fwd(d, p, len, 0);
  uint32_t last_match = 0;  // masks of this state are already in acc
  auto consume = [&](uint32_t ns) {
    s = ns;
    if (s >= d.match_lo && s != last_match) {
      last_match = s;
#pragma unroll
      for (uint32_t w = 0; w < kMaxMaskWords; w++)
        if (w < mw) acc[w] |= d.masks[(uint64_t)s * mw + w];
    }
  };
  // the record 16 bytes at a time (three aligned 8-byte loads) while that stays inside the buffer
  const bool aligned = (reinterpret_cast<uintptr_t>(text) & 7) == 0;
  const uint8_t* const buf_hi = text + offsets[n_rec];
  uint64_t q = 0;
  while (q < len && s != 0) {
    const uint8_t* wp = p + q;
    const uint8_t* al = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(wp) & ~(uintptr_t)7);
    if (aligned && al + 24 <= buf_hi) {
      uint32_t v[4];
      window16(wp, v);
      const uint32_t nb = len - q >= 16 ? 16u : (uint32_t)(len - q);
#pragma unroll
      for (int i = 0; i < 16; i++)
        if ((uint32_t)i < nb && s != 0) consume(T.step(s, window_byte(v, i)));
      q += nb;
    } else {
      consume(T.step(s, p[q]));
      q++;
    }
  }
  if (s != 0) consume(T.step_eof(s));
}

__global__ void set_matches_batch(BatchArgs a) {
  const Table T = stage_table(a.fwd, g_smem, a.use_smem);
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (r >= a.n_rec) return;
  uint64_t acc[kMaxMaskWords] = {0, 0, 0, 0};
  set_record_masks(T, a.fwd, a.text, a.offsets, a.n_rec, r, acc);
  const uint32_t mw = a.fwd.mask_words;
#pragma unroll
  for (uint32_t w = 0; w < kMaxMaskWords; w++)
    if (w < mw) a.out_masks[r * mw + w] = acc[w];
}

// A RegexSet in pattern groups: blockIdx.y is the group.  Its bit j is bit lo + j of the record's row; a word that
// two groups share takes an atomic OR, a word the group owns alone a plain store (the rows are zeroed before).
__global__ void set_matches_batch_groups(GroupBatchArgs a) {
  const GroupDesc& g = a.groups[blockIdx.y];
  const Table T = stage_table(g.view, g_smem, g.use_smem);
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (r >= a.n_rec) return;
  uint64_t acc[kMaxMaskWords] = {0, 0, 0, 0};
  set_record_masks(T, g.view, a.text, a.offsets, a.n_rec, r, acc);
  const uint32_t w0 = g.lo / 64, sh = g.lo % 64, w_last = (g.hi - 1) / 64;
  uint64_t* row = a.out_masks + r * a.row_words;
#pragma unroll
  for (uint32_t i = 0; i <= kMaxMaskWords; i++) {
    const uint32_t k = w0 + i;
    if (k > w_last) break;
    uint64_t v = i < kMaxMaskWords ? acc[i % kMaxMaskWords] << sh : 0;
    if (sh && i > 0) v |= acc[i - 1] >> (64 - sh);
    const bool owned = g.lo <= 64 * k && g.hi >= min(64 * k + 64, a.n_patterns);
    if (owned) row[k] = v;
    else if (v) atomicOr(reinterpret_cast<unsigned long long*>(row + k), (unsigned long long)v);
  }
}


// ---------------------------------------------------------- candidate starts --
// Candidate-start mode (DESIGN.md §2): patterns whose unanchored automata exceed the table budget.  Every
// position whose first min(min_len, 4) bytes lie in the byte sets of the anchored automaton is a candidate
// start; the anchored automaton (kind 0) decides each, so the candidates only need to be a superset of the
// match starts.

// s is a candidate of a text of n bytes (cm: shared-memory byte masks, bit d = in the set of offset d)
__device__ __forceinline__ bool cand_at(const uint8_t* cm, uint32_t depth, const uint8_t* t, uint64_t n, uint64_t s) {
  for (uint32_t d = 0; d < depth; d++)
    if (s + d >= n || !((cm[t[s + d]] >> d) & 1u)) return false;
  return true;
}

// The start bitmap in scan_rev's format.  One thread per bitmap word (64 positions): the 80 bytes
// [64w, 64w + 80) come in as five 16-byte loads where they lie inside the haystack, the masks are looked up in
// shared memory, and the 32 words of a warp are 256 consecutive bytes, so the stores leave as whole sectors.
__global__ void cand_bitmap(const uint8_t* text, uint64_t n, uint64_t base, uint64_t limit, int text_continues, CandArgs c,
                            uint64_t* bitmap, uint8_t* flag0) {
  __shared__ uint8_t cm[256];
  for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) cm[i] = c.mask[i];
  __syncthreads();
  const uint32_t depth = c.depth;
  const bool vec = (reinterpret_cast<uintptr_t>(text) & 15) == 0;
  const uint32_t past_end = text_continues ? 0xFu : 0u;  // a shard's halo ends at n: the text goes on
  const uint64_t w_lo = base >> 6, w_hi = max((limit + 63) >> 6, w_lo + (base == 0 ? 1 : 0));  // word 0 also sets *flag0
  for (uint64_t w = w_lo + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < w_hi; w += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t at = w << 6;  // bit k of word w <-> position at + 1 + k
    uint64_t m0 = 0, m1 = 0, m2 = 0, m3 = 0, cont = 0;
    // byte at + j (j = 1..67) in the set of offset d marks position at + j - d
    auto take = [&](int j, uint32_t raw, bool inside) {
      const uint32_t t = inside ? (uint32_t)cm[raw] : past_end;
      if (j <= 64) { m0 |= (uint64_t)(t & 1u) << (j - 1); if (inside && (raw & 0xC0u) == 0x80u) cont |= 1ull << (j - 1); }
      if (j >= 2 && j <= 65) m1 |= (uint64_t)((t >> 1) & 1u) << (j - 2);
      if (j >= 3 && j <= 66) m2 |= (uint64_t)((t >> 2) & 1u) << (j - 3);
      if (j >= 4) m3 |= (uint64_t)((t >> 3) & 1u) << (j - 4);
    };
    if (vec && at + 80 <= n) {
      uint4 v[5];
#pragma unroll
      for (int i = 0; i < 5; i++) v[i] = ldg128(text + at + 16 * i);
#pragma unroll
      for (int j = 1; j < 68; j++) take(j, word_byte(v[j >> 4], j & 15), true);
    } else {
#pragma unroll 1
      for (int j = 1; j < 68; j++) take(j, at + j < n ? text[at + j] : 0u, at + j < n);
    }
    uint64_t word = ~0ull;
    if (depth > 0) word &= m0;
    if (depth > 1) word &= m1;
    if (depth > 2) word &= m2;
    if (depth > 3) word &= m3;
    if (c.utf8_boundaries) word &= ~cont;
    if (at + 64 > limit) word &= limit > at ? ~0ull >> (64 - (limit - at)) : 0ull;  // positions up to limit
    bitmap[w] = word;
    if (at == 0) {  // position 0 has no bit
      bool hit = true;
      for (uint32_t d = 0; d < depth; d++)
        if (d < n ? !((cm[text[d]] >> d) & 1u) : !text_continues) hit = false;
      if (c.utf8_boundaries && n > 0 && (text[0] & 0xC0u) == 0x80u) hit = false;
      *flag0 = hit;
    }
  }
}

// shortest_match from candidate starts: one lane per segment of seg positions runs the anchored automaton from
// each of its candidates s below the best end known so far and stops at the first match state (before the
// first Match nothing is cut, so that is the earliest end of any match from s).
__global__ void cand_shortest(DfaView fwd, int use_smem, CandArgs c, const uint8_t* text, uint64_t n, uint64_t lo, uint64_t hi,
                              uint32_t seg, unsigned long long* best, int text_continues, uint32_t* overflow) {
  __shared__ uint8_t cm[256];
  for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) cm[i] = c.mask[i];
  __syncthreads();
  const Table T = stage_table(fwd, g_smem, use_smem);
  const uint64_t n_seg = (hi - lo + seg - 1) / seg;
  for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < n_seg; t += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t b = *(volatile unsigned long long*)best;
    const uint64_t s_lo = lo + t * seg, s_hi = min(s_lo + seg, hi);
    for (uint64_t s = s_lo; s < s_hi && s < b; s++) {
      if ((s & 255) == 0) b = min(b, (uint64_t)*(volatile unsigned long long*)best);
      if (!cand_at(cm, c.depth, text, n, s)) continue;
      const uint64_t e = earliest_end(fwd, T, text, n, s, b, text_continues ? overflow : nullptr);
      if (e != kNone) {
        b = e;
        atomicMin(best, (unsigned long long)e);
      }
    }
  }
}

// Batched records from candidate starts, one thread per record (class-indexed tables, the anchored one in shared
// memory when it fits).  find_at(q) = (s*, A(s*)) with s* the first candidate >= q at which the anchored automaton
// finds a match A(s*); with look-arounds the start comes from the reverse-on-slice rule (SURVEY H1) instead.
template <int MODE>
__global__ void batch_cand(BatchArgs a, CandArgs c) {
  __shared__ uint8_t cm[256];
  for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) cm[i] = c.mask[i];
  __syncthreads();
  const Table T = stage_table(a.fwd, g_smem, a.use_smem);
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;  // multiple of 32: warps stay on one ballot word
  const uint32_t lane = threadIdx.x & 31;
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r - lane < a.n_rec; r += stride) {
    bool hit = false;
    uint64_t ms = 0, me = 0;
    if (r < a.n_rec) {
      const uint64_t lo = a.offsets[r], len = a.offsets[r + 1] - lo;
      const uint8_t* p = a.text + lo;
      auto is_cand = [&](uint64_t s) {
        return cand_at(cm, c.depth, p, len, s) && !(c.utf8_boundaries && s < len && (p[s] & 0xC0u) == 0x80u);
      };
      if (MODE == 0) {
        for (uint64_t s = 0; s <= len && !hit; s++)
          hit = is_cand(s) && earliest_end(a.fwd, T, p, len, s) != kNone;
      } else {
        uint64_t s_star = 0;
        auto fwd = [&](uint64_t q) -> uint64_t {  // end of the match at the first candidate >= q that starts one
          for (uint64_t s = q; s <= len; s++) {
            if (!is_cand(s)) continue;
            const uint64_t e = anchored_end(a.fwd, T, p, len, s);
            if (e != kNone) { s_star = s; return e; }
          }
          return kNone;
        };
        auto rev = [&](uint64_t q, uint64_t e) -> uint64_t { return c.slice_rule ? slice_start(a.rev, p, len, q, e) : s_star; };
        if (MODE == 1) {
          me = fwd(0);
          if (me != kNone) {
            ms = me == 0 ? 0 : rev(0, me);
            hit = ms != kNone;
          }
          a.out_spans[2 * r] = hit ? ms : 0;
          a.out_spans[2 * r + 1] = hit ? me : 0;
        } else {
          iter_record<MODE - 2>(a, r, p, len, fwd, rev);
        }
      }
    }
    if (MODE <= 1) {
      const uint32_t bits = __ballot_sync(0xffffffffu, hit);
      if (lane == 0) a.out_bits[r >> 5] = bits;
    }
  }
}
template __global__ void batch_cand<0>(BatchArgs, CandArgs);
template __global__ void batch_cand<1>(BatchArgs, CandArgs);
template __global__ void batch_cand<2>(BatchArgs, CandArgs);
template __global__ void batch_cand<3>(BatchArgs, CandArgs);

}  // namespace rbgpu
