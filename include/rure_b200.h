/*
 * rure_b200.h -- bulk / device-resident extension of the rure C ABI.
 *
 * The reference API is one haystack per call (regex-capi/include/rure.h); GPU-
 * sized work needs bulk entry points.  Every function here returns exactly what
 * looping the scalar ABI would return:
 *   rure_b200_find_all        == collecting rure_iter_next until it returns false
 *   rure_b200_is_match_batch  == rure_is_match(re, hay + off[i], off[i+1]-off[i], 0) per record
 *   rure_b200_find_batch      == rure_find(...)  per record (offsets relative to the record)
 *   rure_b200_set_matches_*   == rure_set_matches(...) packed into 64-bit masks
 *   rure_b200_find_iter_batch == collecting rure_iter_next over each record (record-relative offsets)
 *   rure_b200_captures_batch  == rure_find_captures(re, hay + off[i], off[i+1]-off[i], 0, ...) per record
 *   rure_b200_replace_batch   == rure_b200_replace(re, hay + off[i], off[i+1]-off[i], rep, ..., limit, ...) per record
 *   rure_b200_split_batch     == rure_b200_split(re, hay + off[i], off[i+1]-off[i], has_limit, limit, ...) per record
 *   rure_b200_captures_iter_batch == rure_b200_captures_all(re, hay + off[i], off[i+1]-off[i], ...) per record
 * Functions return true on success; on failure rure_b200_last_error() (thread
 * local) describes what went wrong.  A missing GPU is a failure, never a
 * silent CPU fallback.
 *
 * "_device" variants take CUDA device pointers valid on the current device (one
 * process per GPU; select the device with cudaSetDevice / torch.cuda.set_device
 * before the first call on a regex object).
 */
#ifndef REGEX_B200_RURE_B200_H
#define REGEX_B200_RURE_B200_H

#include "rure.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Compile with `Regex` (str) semantics instead of `bytes::Regex`: the implicit
 * unanchored prefix only skips whole UTF-8 scalars and empty matches advance by
 * one scalar (src/compile.rs:381-395, src/exec.rs:335-337).  Haystacks must be
 * valid UTF-8.  flags/options/error as rure_compile. */
rure *rure_b200_compile_str(const uint8_t *pattern, size_t length, uint32_t flags,
                            rure_options *options, rure_error *error);

/* RegexSet with `regex::RegexSet` (str) semantics; see rure_b200_compile_str. */
rure_set *rure_b200_compile_set_str(const uint8_t **patterns, const size_t *patterns_lengths,
                                    size_t patterns_count, uint32_t flags, rure_options *options,
                                    rure_error *error);

/* ---- the scalar searches of rure.h with an error path ----------------------
 * rure_is_match / rure_shortest_match / rure_find / rure_set_is_match cannot report a run-time
 * failure (the reference's never fail) and abort when the GPU search cannot run; these return
 * false then and set rure_b200_last_error().  Results go to *matched / *found / *end / *match. */
bool rure_b200_is_match(rure *re, const uint8_t *haystack, size_t length, size_t start, bool *matched);
bool rure_b200_shortest_match(rure *re, const uint8_t *haystack, size_t length, size_t start,
                              bool *found, size_t *end);
bool rure_b200_find(rure *re, const uint8_t *haystack, size_t length, size_t start, bool *found,
                    rure_match *match);
bool rure_b200_set_is_match(rure_set *set, const uint8_t *haystack, size_t length, size_t start,
                            bool *matched);

/* ---- single haystack ------------------------------------------------------ */
/* Host haystack.  Large haystacks (>= 128 MiB) are uploaded in 64 MiB pieces and each piece
 * is searched while later pieces are still in flight, spans travelling back meanwhile; the
 * result is identical to uploading first (environment RB200_PIPELINE_PIECE=<bytes> changes
 * the piece size, 0 turns the pipeline off).  Pinned host memory gives the full PCIe rate. */
bool rure_b200_find_all(rure *re, const uint8_t *haystack, size_t length, rure_match *out,
                        size_t cap, size_t *n_total);
bool rure_b200_count_all(rure *re, const uint8_t *haystack, size_t length, size_t *n_total);
/* mask_words = (rure_set_len + 63) / 64 */
bool rure_b200_set_matches_mask(rure_set *set, const uint8_t *haystack, size_t length,
                                size_t start, uint64_t *mask_words);

/* ---- replace / split over all matches (bulk forms of src/re_bytes.rs:476-535 replacen and
 * :316-360, :699-749 split / splitn; the span list and the haystack stay on the device) -------
 * rure_b200_replace: every non-overlapping match (the first `limit` when limit > 0) is replaced by
 * `rep`.  expand != 0 expands `$0`, `${0}` and `$$` as src/expand.rs:50-90 does (a reference to
 * a group the pattern does not have expands to nothing; a reference to any other existing group
 * fails: captures beyond group 0 are not computed by this backend); expand == 0 is NoExpand.
 * *out_len receives the length of the result; at most out_cap bytes are written (out may be
 * NULL to ask for the length).  replace_all = limit 0, replace = limit 1.
 * rure_b200_split: the pieces between the matches as (start, end) pairs; has_limit / limit as
 * splitn (limit pieces at most, the last one being the rest of the haystack). */
bool rure_b200_replace(rure *re, const uint8_t *haystack, size_t length, const uint8_t *rep,
                       size_t rep_len, int expand, size_t limit, uint8_t *out, size_t out_cap,
                       size_t *out_len);
bool rure_b200_replace_device(rure *re, const uint8_t *d_haystack, size_t length,
                              const uint8_t *rep /* host */, size_t rep_len, int expand, size_t limit,
                              uint8_t *d_out, size_t out_cap, size_t *out_len);
bool rure_b200_split(rure *re, const uint8_t *haystack, size_t length, int has_limit, size_t limit,
                     rure_match *out, size_t cap, size_t *n_pieces);
bool rure_b200_split_device(rure *re, const uint8_t *d_haystack, size_t length, int has_limit,
                            size_t limit, rure_match *d_out, size_t cap, size_t *n_pieces);

/* ---- capture groups (src/exec.rs:527-590 read_captures_at; rure_find_captures & co in rure.h use
 * the same path).  The DFA path finds each match; one GPU thread per match then runs the
 * reference's NFA simulation with slots (src/pikevm.rs:130-352) over the narrowed window
 * (src/exec.rs:861-875).  slots: 2 * rure_b200_captures_len(re) entries per match -- start, end of
 * every group, SIZE_MAX where a group did not take part. */
size_t rure_b200_captures_len(rure *re);
bool rure_b200_captures(rure *re, const uint8_t *haystack, size_t length, size_t start, bool *found,
                        size_t *slots);
/* every match of find_iter with its groups: slots[min(cap, *n_matches)][2 * n_groups] */
bool rure_b200_captures_all(rure *re, const uint8_t *haystack, size_t length, size_t *slots, size_t cap,
                            size_t *n_matches, size_t *n_groups);

/* ---- batched records: record i = haystack[offsets[i], offsets[i+1]) -------- */
/* out_bits: bit (i % 8) of byte (i / 8); (n_records + 7) / 8 bytes */
bool rure_b200_is_match_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets,
                              size_t n_records, uint8_t *out_bits);
bool rure_b200_find_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets,
                          size_t n_records, rure_match *out, uint8_t *found_bits);
bool rure_b200_set_matches_batch(rure_set *set, const uint8_t *haystack, const uint64_t *offsets,
                                 size_t n_records, uint64_t *out_masks);
/* Every match of every record.  match_offsets: n_records + 1 entries (always complete); the spans of
 * record i are out[match_offsets[i] .. match_offsets[i+1]), record-relative; at most cap are stored,
 * *n_total counts all.  out == NULL / cap == 0: counts and offsets only.  Str mode
 * (rure_b200_compile_str) steps past an empty match by one UTF-8 scalar. */
bool rure_b200_find_iter_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets, size_t n_records,
                               uint64_t *match_offsets, rure_match *out, size_t cap, size_t *n_total);
/* The capture groups of the first match of every record.  slots: n_records * 2 * rure_b200_captures_len(re)
 * entries, record-relative, SIZE_MAX where a group did not take part (every slot of a record without a
 * match); found_bits as rure_b200_find_batch. */
bool rure_b200_captures_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets, size_t n_records,
                              size_t *slots, uint8_t *found_bits);
/* replacen, split / splitn and captures_iter of every record, with the record as the whole haystack.  Each
 * result is CSR-shaped: an offsets array of n_records + 1 entries (always complete, [0] = 0) and a payload of
 * which at most the given capacity is stored, the total always being reported; a NULL payload or a capacity
 * of 0 asks for sizes only.  Str mode steps past an empty match by one UTF-8 scalar.
 * replace: record i's result is out[out_offsets[i] .. out_offsets[i+1]); rep / expand / limit as
 * rure_b200_replace, limit applying to every record (0 = all matches); *out_len = all output bytes. */
bool rure_b200_replace_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets, size_t n_records,
                             const uint8_t *rep, size_t rep_len, int expand, size_t limit,
                             uint64_t *out_offsets, uint8_t *out, size_t out_cap, size_t *out_len);
/* split: record i's pieces (record-relative start, end) are out[piece_offsets[i] .. piece_offsets[i+1]);
 * has_limit / limit as rure_b200_split, per record (limit 0: no pieces; limit 1: the whole record, even an
 * empty one; the last piece is the rest of the record, empty or not). */
bool rure_b200_split_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets, size_t n_records,
                           int has_limit, size_t limit, uint64_t *piece_offsets, rure_match *out, size_t cap,
                           size_t *n_total);
/* captures_iter: record i's matches are rows match_offsets[i] .. match_offsets[i+1] of
 * slots[min(cap, *n_total)][2 * rure_b200_captures_len(re)], record-relative, SIZE_MAX = group absent. */
bool rure_b200_captures_iter_batch(rure *re, const uint8_t *haystack, const uint64_t *offsets, size_t n_records,
                                   uint64_t *match_offsets, size_t *slots, size_t cap, size_t *n_total);

/* ---- device-resident inputs and outputs ----------------------------------- */
bool rure_b200_find_all_device(rure *re, const uint8_t *d_haystack, size_t length, size_t start,
                               rure_match *d_out, size_t cap, size_t *n_total);
bool rure_b200_shortest_match_device(rure *re, const uint8_t *d_haystack, size_t length,
                                     size_t start, bool *found, size_t *end);
bool rure_b200_set_matches_device(rure_set *set, const uint8_t *d_haystack, size_t length,
                                  size_t start, uint64_t *mask_words /* host */);
/* d_out_bits: 32-bit ballot words, 4 * ((n_records + 31) / 32) bytes of device memory */
bool rure_b200_is_match_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                     size_t n_records, uint32_t *d_out_bits);
bool rure_b200_find_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                 size_t n_records, rure_match *d_out, uint32_t *d_found_bits);
bool rure_b200_set_matches_batch_device(rure_set *set, const uint8_t *d_haystack,
                                        const uint64_t *d_offsets, size_t n_records,
                                        uint64_t *d_out_masks);
/* as rure_b200_find_iter_batch; d_match_offsets and d_out in device memory, *n_total on the host */
bool rure_b200_find_iter_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                      size_t n_records, uint64_t *d_match_offsets, rure_match *d_out,
                                      size_t cap, size_t *n_total);
/* as rure_b200_captures_batch; d_found_bits are 32-bit ballot words as rure_b200_find_batch_device */
bool rure_b200_captures_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                     size_t n_records, size_t *d_slots, uint32_t *d_found_bits);
/* as the three calls above; d_* in device memory (rep stays on the host), totals on the host */
bool rure_b200_replace_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                    size_t n_records, const uint8_t *rep, size_t rep_len, int expand,
                                    size_t limit, uint64_t *d_out_offsets, uint8_t *d_out, size_t out_cap,
                                    size_t *out_len);
bool rure_b200_split_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                  size_t n_records, int has_limit, size_t limit, uint64_t *d_piece_offsets,
                                  rure_match *d_out, size_t cap, size_t *n_total);
bool rure_b200_captures_iter_batch_device(rure *re, const uint8_t *d_haystack, const uint64_t *d_offsets,
                                          size_t n_records, uint64_t *d_match_offsets, size_t *d_slots,
                                          size_t cap, size_t *n_total);

/* ---- byte-range shards of one haystack (multi-GPU; one process per GPU) ------
 * Each rank holds [left context | owned bytes | right halo] of the haystack in its
 * own HBM and searches it with the call below; the ranks exchange only the three
 * boundary values marked (x) -- see regex_b200/sharded.py for the protocol:
 *   rev_left  -> left neighbour's rev_entry   (reverse-scan state at the shared edge)
 *   exit_p/lm -> right neighbour's chain_p/lm (find_iter iterator state)
 *   n_matches -> all ranks (global output offsets)
 * Positions are relative to the buffer; own_lo and own_hi are multiples of 256
 * (own_lo = 0 for the first shard, own_hi = n_buf for the last). */
#define RURE_B200_NO_STATE 0xFFFFFFFFu
#define RURE_B200_NONE (~(uint64_t)0)
#define RURE_B200_SPEC (~(uint64_t)0 - 1)
typedef struct rure_b200_shard {
  /* in */
  uint64_t own_lo, own_hi; /* owns match starts at positions (own_lo, own_hi] (+ 0 for the first shard) */
  int32_t is_first, is_last;
  uint32_t rev_entry;      /* (x) exact state at own_hi, or RURE_B200_NO_STATE to speculate */
  uint32_t reuse_scan;     /* keep the start bitmap computed by the previous call on this buffer */
  uint64_t chain_p, chain_lm; /* (x) iterator state entering the shard, or RURE_B200_SPEC */
  /* out */
  uint32_t rev_guess;      /* state the scan assumed at own_hi */
  uint32_t rev_left;       /* (x) exact state at own_lo */
  uint64_t exit_p, exit_lm;   /* (x) iterator state leaving the shard */
  uint64_t n_matches;      /* (x) */
  uint32_t halo_overflow;  /* call failed: bit 0 = a match ran past the end of the right halo, bit 1 = the
                              reverse-on-slice scan of a look-around pattern reached a clamped chain_p (left context too short) */
  uint32_t chain_clamped;  /* in: chain_p is the buffer position standing in for a restart point LEFT of the buffer */
} rure_b200_shard;
bool rure_b200_find_all_shard_device(rure *re, const uint8_t *d_buffer, size_t n_buffer,
                                     rure_b200_shard *io, rure_match *d_out, size_t cap);

/* is_match / shortest_match / RegexSet::matches over one shard (positions [own_lo, own_hi) of the
 * buffer; the last shard also takes the end-of-text step).  The forward automaton's state flows
 * left to right: entry_state is the left neighbour's exact exit_state, or RURE_B200_NO_STATE to
 * guess it from the left context; regex_b200/sharded.py (forward_sharded) compares entry_used
 * with the neighbour's exit_state and searches again on a mismatch.  Results: first_end = end of
 * the first match that ends in this shard (buffer-relative; shortest_match = min over ranks),
 * masks = patterns that match inside it (RegexSet::matches = OR over ranks; 4 words = 256 patterns).
 * rure_b200_set_matches_shard_device returns false with a message for a set searched in pattern
 * groups (see rure_b200_set_groups): one entry state and 256 mask bits cannot describe it. */
typedef struct rure_b200_fwd_shard {
  /* in */
  uint64_t own_lo, own_hi;
  int32_t is_first, is_last;
  uint32_t entry_state;
  /* out */
  uint32_t entry_used, exit_state, found;
  uint64_t first_end;
  uint64_t masks[4];
} rure_b200_fwd_shard;
bool rure_b200_shortest_match_shard_device(rure *re, const uint8_t *d_buffer, size_t n_buffer,
                                           rure_b200_fwd_shard *io);
bool rure_b200_set_matches_shard_device(rure_set *set, const uint8_t *d_buffer, size_t n_buffer,
                                        rure_b200_fwd_shard *io);

/* ---- threads ----------------------------------------------------------------
 * As in rure.h (regex-capi/include/rure.h:27-34) one compiled rure / rure_set may be used from
 * several threads at once.  The scalar entry points (rure_is_match, rure_find, rure_shortest_match,
 * rure_find_captures, rure_set_is_match, rure_set_matches and their rure_b200_* twins with an error
 * return) run concurrently: the engine keeps its device scratch per object, so a call that finds the
 * object busy runs on a clone compiled from the same source, kept with the handle.  The bulk,
 * device-pointer and shard entry points use the handle's primary engine and serialise; give every
 * thread (or shard) its own handle for those.  rure_b200_last_stats* and the options describe the
 * primary engine. */
/* ---- diagnostics ----------------------------------------------------------- */
const char *rure_b200_last_error(void);
/* kernels launched by this library in this process (bench.py "gpu_launches") */
uint64_t rure_b200_kernel_launches(void);
/* Timing (CUDA events on the library's stream) and fix-up counters of the last
 * rure_b200_find_all* call on this object.  out[0..7] = scan_ms, walk_ms,
 * total_ms, scan_redo_rounds, scan_redo_segments, stitch_rounds, stitch_dirty_chunks,
 * fused (1 when the scan kernel also walked the chains, so scan_ms covers both) */
void rure_b200_last_stats(rure *re, double *out8);
/* The same plus out[8..11] = sequential stitch passes, state-map passes (segments run from
 * every boundary state), waves of the last forward search, path of the last find_all
 * (0 generic scan, 1 fast scan, 2 fused scan+walk, 3 literal prefilter, 4 candidate starts: a pattern whose
 * unanchored automata exceed the DFA budget, searched with the anchored one), out[12] = matches longer
 * than 256 KiB that were measured by the parallel long-run pass.  n = doubles to write. */
void rure_b200_last_stats_ex(rure *re, double *out, size_t n);
/* rure_b200_set_last_stats_ex also has out[13] = pattern groups searched in the first wave of the last
 * set call (1 = the product automaton; see rure_b200_set_groups). */
void rure_b200_set_last_stats_ex(rure_set *set, double *out, size_t n);
/* Named knobs (tests, tuning): "wave0" bytes of the first wave of is_match / shortest_match /
 * set matches (x16 per wave, 0 = one wave), "narrow_sets" 0/1, "max_stitch_rounds",
 * "max_redo_rounds", "batch_refill" 0/1 (batched is_match: lanes refill from a task of records), "prefilter" (0 never, 1 automatic: only for a single rare byte, 2 whenever the
 * pattern qualifies), "candidate_starts" 0/1 (tests: search from candidate starts with the anchored
 * automaton, as patterns over the DFA budget do, even when the unanchored automata fit).
 * Returns false for an unknown name.
 * Sets also take "set_group_patterns" k (tests): search in groups of at most k patterns even when
 * the product automaton fits, each group split further while its automaton is over the budget;
 * 0 (the default) = automatic.  The new plan is compiled at once; false when a group fails to compile
 * (the plan is then unchanged). */
bool rure_b200_set_option(rure *re, const char *name, uint64_t value);
bool rure_b200_set_set_option(rure_set *set, const char *name, uint64_t value);
/* RegexSets of any size.  A set of at most 256 patterns whose forward all-match automaton fits the DFA
 * budget is searched with that one product automaton.  Larger sets, and sets whose product automaton is
 * over the budget, are searched in pattern groups: contiguous pattern ranges of at most 256 patterns, each
 * with its own automaton within the budget (chunks of 256, halved while over the budget, on multiples of
 * 64 above 64 patterns).  A single pattern over the budget is still a compile error.  Every set call
 * answers the same either way; rure_set_matches takes any set size.  Returns the number of groups (1 for
 * the product automaton, 0 for an empty set) and writes the first pattern index of up to cap of them to first_pattern
 * (may be NULL). */
size_t rure_b200_set_groups(rure_set *set, size_t *first_pattern, size_t cap);
/* seg/chunk are positions per scan segment / walk chunk (multiples of 64);
 * warm = warm-up bytes (0 = automatic); 0 keeps the current value elsewhere. */
void rure_b200_set_tuning(rure *re, uint32_t seg, uint32_t chunk, uint32_t warm, uint32_t block,
                          uint32_t blocks_per_sm);
/* Launch this object's kernels on a caller-owned cudaStream_t (e.g. torch's current
 * stream) instead of its private stream; pass the stream handle as a pointer value. */
void rure_b200_set_stream(rure *re, void *cuda_stream);
void rure_b200_set_set_stream(rure_set *set, void *cuda_stream);
/* Tests: route scans through the generic kernel even when the fast one applies. */
void rure_b200_force_generic(rure *re, int yes);
/* Walk each segment's find_iter chain inside the fast scan kernel (default on). */
void rure_b200_set_fuse(rure *re, int yes);
/* Feed the fast scan kernel with 2-D tiled TMA box loads (default on; off = per-lane bulk copies). */
void rure_b200_set_tensor_tma(rure *re, int yes);
/* Dense tables, for tests and tooling.  kind: 0 forward anchored leftmost-first,
 * 1 reverse unanchored all-match, 2 forward unanchored all-match, 3 reverse
 * anchored longest, 4 forward unanchored leftmost-first.  A pattern searched from candidate
 * starts has kinds 0 and 3 only: kinds 1, 2 and 4 return false with a message.  Kind 2 of a set
 * searched in pattern groups returns false with a message that lists the groups.
 * info[0..5] = n_states, n_classes (last = EOF), match_lo, mask_words, uniform_start, raw_states.
 * Buffers may be NULL to query sizes: trans n_states*n_classes u16, classes 256 u8,
 * start 128 u16, masks n_states*mask_words u64. */
bool rure_b200_dfa_export(rure *re, int kind, uint32_t *info6, uint16_t *trans, uint8_t *classes,
                          uint16_t *start, uint64_t *masks);
/* info[0..3] = min match length, max match length (SIZE_MAX = unbounded), can_match_empty, has_looks */
void rure_b200_pattern_info(rure *re, uint64_t *info4);

#ifdef __cplusplus
}
#endif
#endif
