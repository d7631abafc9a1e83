// Kernel argument blocks + declarations shared by kernels.cu and engine.cu.
#pragma once
#include <cstdint>
#include <cuda.h>

#include "kernels.cuh"

namespace rbgpu {

constexpr uint32_t kMaxMaskWords = 4;  // RegexSet of up to 256 patterns per scan
constexpr uint32_t kNoEntry = 0xFFFFFFFFu;

struct ScanArgs {
  DfaView dfa;
  int use_smem;
  const uint8_t* text;
  uint64_t n;        // haystack (buffer) length
  uint64_t limit;    // reverse scan: bytes [base, limit) are scanned (== n except for shards)
  uint64_t base;     // first position covered (64-aligned for bitmap scans)
  uint64_t n_seg;
  uint32_t seg;      // positions per segment (multiple of 64)
  uint32_t warm;     // warm-up bytes for the speculative entry state
  uint64_t* bitmap;  // reverse scan: bit i <=> a match starts at position i+1
  uint8_t* flag0;    // reverse scan: a match starts at position 0
  HotView hot;              // fast kernels: byte-indexed table over the hot states
  uint64_t tmap_rows;       // fast kernels: rows (full segments) covered by the 2-D tensor map, 0 = none
  uint64_t* seg_first;  // forward scan: first match end per segment
  uint64_t* seg_mask;   // forward scan: OR of masks per segment (nullable)
  uint16_t* guess;
  uint16_t* fin;
  const uint32_t* redo_list;  // nullable: only these segments, entry = neighbour's fin
  const uint32_t* n_redo;
  int utf8_boundaries;  // drop starts that are not UTF-8 scalar boundaries (Regex on str)
  uint64_t skip_lo, skip_hi;  // scan_fwd_reduce: segments [skip_lo, skip_hi) belong to scan_fwd_fast
  uint64_t fwd_limit;   // forward scan: positions [base, fwd_limit) are stepped; n + 1 includes the end-of-text step
  uint32_t entry0;      // forward scan: exact state at `base` (a later wave of one search), kNoEntry = start state by flags
  uint32_t tbase_off, fbase_off;  // scan_rev_fast: row 0 of the reverse table and the forward table, in bytes from the ring base (host-computed:
                                  // derived from the table sizes in the kernel they were recomputed for every 16 haystack bytes)
};

struct WalkArgs {
  DfaView fwd;  // forward, anchored, leftmost-first
  DfaView rev;  // reverse, anchored, longest (reference dfa_reverse) -- slice emulation only
  const uint8_t* text;
  uint64_t n;
  uint64_t limit;        // candidate bits [base, limit) (== n except for shards)
  int text_continues;    // shard: the haystack goes on after n (no EOF there)
  uint32_t* err_flag;    // set when a match runs past the end of a shard's halo
  uint64_t clamp_p;      // shard entered at a restart point left of its buffer: the buffer position standing in for it (else kNone)
  uint32_t* floor_flag;  // set when a reverse-on-slice scan from clamp_p's match reaches clamp_p alive (left context too short)
  const uint64_t* bitmap;
  const uint8_t* flag0;
  uint64_t base;  // first bitmap bit of chunk 0 (64-aligned); bit i <-> position i+1
  uint64_t n_chunks;
  uint32_t chunk;  // bitmap bits per chunk (multiple of 256)
  uint32_t stage_cap;  // staged spans per chunk
  uint64_t* stage;     // [n_chunks][stage_cap] spans
  int use_smem;
  uint64_t* first_cand;  // per chunk: position of its first candidate (kNone if none)
  uint64_t* in_p;
  uint64_t* in_lm;
  uint64_t* out_p;
  uint64_t* out_lm;
  uint64_t* count;          // per chunk: spans it contributes to the output (after trimming / covering)
  const uint64_t* offset;
  uint32_t* skip;           // per chunk: staged spans dropped from the front by the stitch (trimmed speculation)
  uint32_t* meta;           // per chunk: spans the walk produced (bits 0-28, may exceed stage_cap) | kMetaPatched | chunk state << 30
  uint32_t* dirty_list;     // chunks to walk again (nullable: all chunks)
  const uint32_t* n_dirty;
  uint64_t seq_from;        // walk_sequential: first chunk of the sequential pass
  uint64_t exact_cap;       // longest anchored run a chunk walked from its exact entry does itself (kNone = any)
  const uint64_t* long_tab; // n_long (start, end) pairs of long matches measured by the host-driven parallel scan
  uint32_t n_long;
  unsigned long long* long_req;  // smallest start whose run exceeded exact_cap (kNone = none): the host resolves it next
  HotView fwd_hot;              // fast runner: byte-indexed forward anchored table (hot states)
  uint64_t fixed_len;           // fixed-length runner: every match has this many bytes
  uint64_t* out;  // spans: start, end pairs
  uint64_t cap;
  int utf8;
  int emulate_slice;
  int can_match_empty;
};

// Literal prefilter (kernels.cu "literal prefilter"): the byte to scan for and the byte sets a
// match can have at its first offsets, derived from the anchored forward automaton on the host.
struct PfArgs {
  uint32_t o;           // offset of the scanned byte inside a match (< min match length)
  uint32_t n_bytes;     // 1..4 byte values to scan for
  uint32_t bcast[4];    // each replicated into the four bytes of a word
  uint32_t n_sets;      // leading offsets 0..n_sets-1 of a match with a membership set (<= 4)
  uint32_t sets[4][8];  // 256-bit sets
};
// mode 0: every chunk (one warp per chunk, grid-stride); 1: the dirty list; 2: sequential pass from
// a.seq_from (one warp); 3: chunks that overflowed their staging slots, straight into a.out
template <int FAST, int NB>  // NB = PfArgs::n_bytes
__global__ void literal_scan(const __grid_constant__ WalkArgs a, const __grid_constant__ PfArgs pf, int mode);
__global__ void compact_staged(WalkArgs a);

// Candidate-start mode (DESIGN.md §2): position s is a candidate when text[s + d] is in the byte set of offset d for
// every d < depth (the bytes with which some start state of the anchored automaton survives d + 1 steps).
// Candidates are a superset of the match starts; the anchored automaton decides each.
struct CandArgs {
  uint32_t depth;        // min(min_len, 4); 0 = every position is a candidate, n included
  int utf8_boundaries;   // as ScanArgs: drop positions inside a UTF-8 sequence (Regex on str, empty matches)
  int slice_rule;        // batched find: the start of a match comes from the reverse-on-slice scan (look-arounds)
  uint8_t mask[256];     // bit d set when the byte is in the set of offset d
};
// bitmap bits [base, limit) (bit i <-> position i + 1) and, when base == 0, *flag0 (position 0); base is 64-aligned.
// text_continues: a shard's halo ends at n, positions whose sets reach past it stay candidates
__global__ void cand_bitmap(const uint8_t* text, uint64_t n, uint64_t base, uint64_t limit, int text_continues, CandArgs c,
                            uint64_t* bitmap, uint8_t* flag0);
// *best = min(*best, the first position where the anchored automaton, started at a candidate s in [lo, hi), enters a
// match state); one lane per seg positions.  text_continues: the text goes on after n (a stream's window); a run that
// reaches n undecided sets *overflow.
__global__ void cand_shortest(DfaView fwd, int use_smem, CandArgs c, const uint8_t* text, uint64_t n, uint64_t lo, uint64_t hi,
                              uint32_t seg, unsigned long long* best, int text_continues, uint32_t* overflow);

// ---- bulk operations over the span list (src/re_bytes.rs:316-360 split, :476-535 replacen) ----
// The replacement of one match is a sequence of parts: literal bytes, or the text of a capture
// group of that match (`$0`, `$2`, `$name`; src/expand.rs:50-90).
constexpr uint32_t kMaxRepParts = 16;
constexpr uint32_t kRepGroup = 0x80000000u;  // part_len = kRepGroup | group index
struct ReplaceArgs {
  const uint8_t* text;
  uint64_t n;
  const uint64_t* spans;   // n_matches (start, end) pairs, ordered, non-overlapping
  uint64_t n_matches;      // matches to replace (after `limit`)
  const uint64_t* lens_before;  // exclusive prefix sum of the match lengths
  const uint64_t* reps_before;  // exclusive prefix sum of the replacement lengths
  const uint64_t* slots;   // [n_matches][n_slots] group spans (null when only group 0 is referenced)
  uint32_t n_slots;
  const uint8_t* lits;     // literal bytes of all parts, concatenated
  uint32_t n_parts;
  uint32_t part_len[kMaxRepParts];  // literal length, or kRepGroup | g
  uint32_t part_off[kMaxRepParts];  // offset into lits
  uint64_t lit_total;      // literal bytes per match
  uint8_t* out;
  uint64_t out_cap;
};
__global__ void replace_lengths(ReplaceArgs a, uint64_t* rep_lens);
__global__ void span_lengths(const uint64_t* spans, uint64_t n_matches, uint64_t* lens);
// words[i] += add (window-relative spans of a stream -> stream offsets)
__global__ void add_to_words(uint64_t* words, uint64_t n, uint64_t add);
__global__ void replace_gaps(ReplaceArgs a, uint64_t matched_total, uint64_t replaced_total);
__global__ void replace_matches(ReplaceArgs a);
// pieces[i] = text between match i-1 and match i; limit as splitn (0 = none)
__global__ void split_pieces(const uint64_t* spans, uint64_t n_matches, uint64_t n, uint64_t n_pieces, int last_is_rest, uint64_t* pieces, uint64_t cap);

// ---- batched records: replacen / splitn / captures_iter per record (engine.cu *_batch_device) ----
// A CSR list (csr[n_rec + 1], csr[0] = 0) gives the items of record r at [csr[r], csr[r + 1]); spans are record-relative.
// counts[r] = min(csr[r + 1] - csr[r], limit), counts[n_rec] = 0 (ready for an exclusive scan into a new CSR)
__global__ void csr_counts(const uint64_t* csr, uint64_t n_rec, uint64_t limit, uint64_t* counts);
// the first kcsr[r + 1] - kcsr[r] spans of every record, compacted to kept[kcsr[r] ..)
__global__ void batch_keep_spans(const uint64_t* csr, const uint64_t* kcsr, uint64_t n_rec, const uint64_t* spans, uint64_t m, uint64_t* kept);
// record-relative -> relative to offsets[0]: spans and, when slots is not null, every group slot that took part
__global__ void batch_to_base(const uint64_t* offsets, const uint64_t* csr, uint64_t n_rec, uint64_t* spans, uint64_t m, uint64_t* slots,
                              uint32_t n_slots);
// out_offsets[r] = (offsets[r] - offsets[0]) - L[csr[r]] + P[csr[r]]; L / P = lens_before / reps_before extended by the totals
__global__ void batch_replace_offsets(const uint64_t* offsets, const uint64_t* csr, uint64_t n_rec, const uint64_t* lens_before,
                                      const uint64_t* reps_before, uint64_t m, uint64_t matched_total, uint64_t replaced_total,
                                      uint64_t* out_offsets);
// pieces of every record as split_device counts them (counts[n_rec] = 0); has_limit / limit as splitn
__global__ void batch_split_counts(const uint64_t* offsets, const uint64_t* csr, const uint64_t* spans, uint64_t n_rec, int has_limit,
                                   uint64_t limit, uint64_t* counts);
// piece i < n_out of the piece CSR pcsr, record-relative (split_pieces of its record)
__global__ void batch_split_pieces(const uint64_t* offsets, const uint64_t* csr, const uint64_t* spans, const uint64_t* pcsr, uint64_t n_rec,
                                   int has_limit, uint64_t limit, uint64_t* pieces, uint64_t n_out);
// records where the NFA's group 0 of some match differs from its find_iter span: bit r of flags (zeroed before) set
// once, r appended to list[*n_list]
__global__ void batch_diverged(const uint64_t* csr, uint64_t n_rec, const uint64_t* spans, uint64_t m, const uint64_t* slots, uint32_t n_slots,
                               uint32_t* flags, uint64_t* list, unsigned int* n_list);
// rows (width words) of the records whose bit in skip is clear, from their place in csr to their place in new_csr
// (rows at or beyond cap are dropped)
__global__ void batch_move_rows(const uint64_t* csr, const uint64_t* new_csr, uint64_t n_rec, const uint32_t* skip, const uint64_t* src, uint64_t m,
                                uint32_t width, uint64_t* dst, uint64_t cap);

// ---- capture groups on the narrowed window (src/exec.rs:861-875, src/pikevm.rs:130-352) ----
struct NfaInst { uint32_t op_look_lo_hi; uint32_t a, b; };  // op | look << 8 | lo << 16 | hi << 24; a, b as rb::Inst
struct CapArgs {
  const NfaInst* insts;
  uint32_t n_insts, start_ip, n_slots;
  int anchored_start;      // the pattern begins with ^ (no lazy prefix, no later threads)
  const uint8_t* text;
  uint64_t n;
  const uint64_t* spans;   // (start, end) of every match, from the DFA path
  uint64_t n_matches;
  uint64_t* slots;         // [n_matches][n_slots], kNone = the group did not take part
  uint8_t* scratch;        // per resident thread: two thread lists with their slot arrays, a stack (see kernels.cu)
  uint64_t per_thread;
  // batched records (null otherwise): match m is the first match of record m, spans are record-relative and
  // the record is the text; records whose bit in rec_found (ballot words) is clear are skipped
  const uint64_t* rec_offsets;
  const uint32_t* rec_found;
  // batched records with any number of matches each (null otherwise; rec_found is then unused): match m belongs
  // to the record r with rec_csr[r] <= m < rec_csr[r + 1] (n_rec + 1 entries)
  const uint64_t* rec_csr;
  uint64_t n_rec;
};
__global__ void pike_captures(CapArgs a);
// ballot words: bit r = group 0 of record r took part (slots[r * n_slots] != kNone)
__global__ void slot_found_bits(const uint64_t* slots, uint32_t n_slots, uint64_t n_rec, uint32_t* bits);

struct BatchArgs {
  DfaView fwd;
  DfaView rev;
  HotView fwd_hot, rev_hot;          // batch_fast: byte-indexed hot tables
  const DfaView* fwd_g;              // the same views in global memory (cold fallback)
  const DfaView* rev_g;
  int use_smem;
  const uint8_t* text;
  const uint64_t* offsets;  // n_rec + 1
  uint64_t n_rec;
  uint32_t* out_bits;   // ballot words
  uint64_t* out_spans;  // 2 per record
  uint64_t* out_masks;  // mask_words per record
  unsigned long long* task_counter;  // batch_refill: next task to hand out (zeroed before the launch)
  uint32_t task_recs;                // batch_refill: records per task (multiple of 32, <= 2048)
  // batch_iter*: per-record find_iter
  uint64_t* match_offsets;  // count pass: matches of record r at [r]; write pass: exclusive prefix sum (first slot of record r)
  uint64_t cap;             // write pass: spans stored at out_spans[0, cap)
  int utf8;                 // empty matches advance by one UTF-8 scalar (Regex on str)
  int fwd_only;             // count pass of a pattern that cannot match empty and has no look-around: no reverse scan
};

template <int MODE>
__global__ void batch_fast(BatchArgs a);
// PASS 0: count the matches of every record; PASS 1: write them.  _fast: hot tables in shared memory.
template <int PASS>
__global__ void batch_iter_fast(BatchArgs a);
template <int PASS>
__global__ void batch_iter(BatchArgs a);
// batched records from candidate starts (fwd = anchored leftmost-first, rev = reverse anchored longest):
// MODE 0 is_match, 1 find, 2 find_iter count pass, 3 find_iter write pass
template <int MODE>
__global__ void batch_cand(BatchArgs a, CandArgs c);
// batched is_match, the lanes of a warp refilled from a task of task_recs records
__global__ void batch_refill(BatchArgs a);
__global__ void scan_rev_bitmap(ScanArgs a);
template <int FUSED>
__global__ void scan_rev_fast(ScanArgs a, WalkArgs wa, const __grid_constant__ CUtensorMap tmap);
__global__ void scan_fwd_reduce(ScanArgs a);
__global__ void scan_fwd_fast(ScanArgs a, const __grid_constant__ CUtensorMap tmap);
__global__ void verify_segments(const uint16_t* guess, const uint16_t* fin, uint64_t n_seg, int reverse,
                                uint32_t* redo_list, uint32_t* n_redo);
// ---- exact segment entry states by state-map composition (bounded fix-up; engine.cu solve_entries) ----
__global__ void mark_states(const uint16_t* a, uint64_t n, uint8_t* present);
// maps[t * k + j] = state after running segment t from states[j]  (reverse: right to left)
__global__ void scan_map(ScanArgs a, int reverse, const uint16_t* states, uint32_t k, uint16_t* maps);
// *n_new += map values that are not in the state list (kidx == 0xFFFF); those are marked in present[]
__global__ void closure_check(const uint16_t* maps, uint64_t n, const uint16_t* kidx, uint8_t* present, uint32_t* n_new);
// blocks of kMapBlock segments: comp[b * k + j] = composite of the block's maps applied to states[j]
constexpr uint32_t kMapBlock = 1024;
__global__ void compose_blocks(const uint16_t* maps, const uint16_t* kidx, const uint16_t* states, uint32_t k, uint64_t n_seg,
                               int reverse, uint16_t* comp);
// one thread: entry state of every block, walking the blocks in scan direction from the exact state `first_entry`
__global__ void compose_top(const uint16_t* comp, const uint16_t* kidx, uint32_t k, uint64_t n_blocks, int reverse,
                            const uint16_t* first_entry, uint16_t* block_entry);
// exact[t] = entry state of segment t
__global__ void compose_fill(const uint16_t* maps, const uint16_t* kidx, uint32_t k, uint64_t n_seg, int reverse,
                             const uint16_t* block_entry, uint16_t* exact);
// neighbour[t -/+ 1] := exact[t] so that verify_segments + one redo round finish the job
__global__ void publish_exact(const uint16_t* exact, uint64_t n_seg, int reverse, uint16_t* fin);
// last position at which the anchored automaton, entered in exact[t], is in a match state inside segment t (+1; 0 = none)
__global__ void scan_last_match(ScanArgs a, const uint16_t* exact, unsigned long long* best, uint32_t* alive_at_end);
__global__ void reduce_segments(const uint64_t* seg_first, const uint64_t* seg_mask, uint64_t n_seg, uint32_t mw,
                                unsigned long long* result);
template <int FAST>
__global__ void walk_chunks(WalkArgs a);
template <int FAST>
__global__ void compact_spans(WalkArgs a);
template <int FAST>
__global__ void walk_sequential(WalkArgs a);
__global__ void init_walk_entries(uint64_t* in_p, uint64_t* in_lm, uint32_t* skip, uint64_t n_chunks, uint64_t p0, uint64_t lm0);
// Chunk states kept in WalkArgs::meta (bits 30-31).
constexpr uint32_t kChunkOk = 0, kChunkIdent = 1, kChunkCovered = 2, kChunkDeferred = 3;
constexpr uint32_t kMetaCount = 0x1FFFFFFFu;
constexpr uint32_t kMetaPatched = 0x20000000u;  // the first staged span's start was re-derived by the slice rule
// One entry of the "exit of the last contributing chunk to the left" scan: key = p + 1 (0 = no
// contribution yet, ~0 = the iteration is over), lm = previous match end that goes with it.
struct ChainKey { uint64_t key, lm; };
// counters: [0] dirty chunks, [1] changed decisions, [2] need the general loop, [3] smallest dirty chunk index
__global__ void stitch_fast(WalkArgs a, uint32_t* counters);
__global__ void entries_local(WalkArgs a, ChainKey* excl, ChainKey* block_tot, uint32_t* first_deferred);
__global__ void entries_blocks(ChainKey* block_tot, uint64_t n_blocks, ChainKey* grand);
__global__ void stitch_resolve(WalkArgs a, const ChainKey* excl, const ChainKey* block_tot, uint32_t* counters);
__global__ void scan_counts_local(const uint64_t* in, uint64_t* out, uint64_t* block_sums, uint64_t n);
__global__ void scan_block_sums(uint64_t* block_sums, uint64_t n_blocks, unsigned long long* grand_total);
__global__ void scan_add_block_offsets(uint64_t* out, const uint64_t* block_sums, uint64_t n);
__global__ void is_match_batch(BatchArgs a);
__global__ void find_batch(BatchArgs a);
__global__ void set_matches_batch(BatchArgs a);
// A RegexSet in pattern groups (engine.cu set_matches_batch_groups): group g owns patterns [lo, hi)
struct GroupDesc {
  DfaView view;
  uint32_t lo, hi;
  int use_smem;  // the group's table is staged in shared memory
};
struct GroupBatchArgs {
  const GroupDesc* groups;  // gridDim.y entries, in global memory
  const uint8_t* text;
  const uint64_t* offsets;  // n_rec + 1
  uint64_t n_rec;
  uint64_t* out_masks;      // row_words per record, zeroed before the launch
  uint32_t row_words;       // (n_patterns + 63) / 64
  uint32_t n_patterns;
};
__global__ void set_matches_batch_groups(GroupBatchArgs a);

}  // namespace rbgpu
