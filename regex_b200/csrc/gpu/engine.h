// Host side of the B200 search backend: owns the determinized tables on the
// device and orchestrates the kernels.  This is the analogue of the reference's
// ExecNoSync (src/exec.rs:365-596): same operations, same results, but every
// search runs on the GPU -- there is no CPU matching path in this library.
#pragma once
#include <cstdint>
#include <algorithm>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../dfa/determinize.h"
#include "../frontend/frontend.h"

namespace rbgpu {

struct BatchArgs;      // launch.h
struct ScanArgs;       // launch.h
struct WalkArgs;       // launch.h
struct ChainKey;       // launch.h
struct DeviceScalars;  // engine.cu
struct HostScalars;    // engine.cu

struct CompileOptions {
  uint32_t flags = 32;               // RURE_FLAG_* bits (rure.h:56-68); default = UNICODE
  size_t size_limit = 10u << 20;     // program size limit (re_builder.rs:29)
  size_t dfa_size_limit = 2u << 20;  // scaled x16 into the dense-table budget (DESIGN.md)
  bool only_utf8 = false;            // false = bytes::Regex, true = Regex (str)
  bool as_set = false;               // RegexSet semantics even for one pattern
};

enum DfaKind { kFwdAnchoredLF = 0, kRevUnanchoredAll, kFwdUnanchoredAll, kRevAnchoredLongest, kFwdUnanchoredLF, kNumDfaKinds };

struct Tuning {
  uint32_t seg = 0;        // bytes per scan segment (multiple of 64); 0 = automatic
  bool force_generic = false;  // tests: use the generic scan kernel even when the fast one applies
  bool fuse = true;            // walk each segment's chain inside the fast scan kernel
  bool tensor_tma = true;      // feed the fast scan kernel with 2-D tiled TMA loads
  uint32_t chunk = 2048;   // bitmap bits per chain-walk chunk (one thread; multiple of 256)
  uint32_t warm = 0;       // 0 = automatic (bounded patterns: max match length; else 128)
  uint32_t block = 256;
  uint32_t blocks_per_sm = 8;
  uint64_t wave0 = 64ull << 20;  // first wave of a forward search in bytes (x16 per wave); 0 = one wave
  bool narrow_sets = true;
  int batch_refill = 1;          // batched is_match: lanes take the next record as soon as theirs is decided (kernels.cu batch_refill) instead of
                                 // one record per lane per round; 0 off, 1 batches large enough for tasks of >= 96 records, 2 any size (tests)
  int prefilter = 1;             // literal_scan instead of the DFA scan: 0 never, 1 when the scanned byte is estimated rare enough
                                 // to win (one byte, <= ~0.12 % of the haystack), 2 whenever the pattern qualifies structurally       // RegexSet::matches: continue with the automaton of the still-unmatched patterns
  uint32_t max_stitch_rounds = 16;  // re-walk rounds before the stitch falls back to one sequential pass
  uint32_t max_redo_rounds = 3;     // scan redo rounds before segment entry states are solved by state-map composition
  bool candidate_starts = false;    // tests: search from candidate starts (as over-budget patterns do) even when the unanchored automata fit
};

struct Stats {  // filled by the last single-haystack call (diagnostics, bench roofline)
  uint64_t scan_redo_rounds = 0, scan_redo_segments = 0;
  uint64_t stitch_rounds = 0, stitch_dirty_chunks = 0, sequential_passes = 0, map_passes = 0, waves = 0, long_runs = 0;
  float scan_ms = 0, walk_ms = 0, total_ms = 0;
  bool fused = false;  // the scan kernel also walked the chains (scan_ms covers both)
  int path = 0;        // last find_all: 0 generic scan, 1 fast scan, 2 fused scan + walk, 3 literal prefilter, 4 candidate starts
  uint32_t groups = 0; // RegexSet calls: pattern groups (automata) searched in the first wave
};

constexpr uint32_t kNoState = 0xFFFFFFFFu;

// One byte-range shard of a larger haystack (multi-GPU, SURVEY.md 8e).  The buffer is
// [left context | owned bytes | right halo]; positions are buffer-relative.
struct ShardIO {
  // in
  uint64_t own_lo = 0, own_hi = 0;  // owns match starts at positions (own_lo, own_hi] (+ position 0 if own_lo == 0)
  bool is_first = true, is_last = true;  // buffer begins / ends where the haystack does
  uint32_t rev_entry = kNoState;    // exact reverse-scan state at own_hi from the right neighbour
  uint64_t chain_p = 0, chain_lm = ~0ull;  // iterator state entering the shard (kSpec = speculate)
  bool reuse_scan = false;          // keep the start bitmap of the previous call on this buffer
  bool chain_clamped = false;       // chain_p stands in for a restart point left of the buffer (look-around patterns:
                                    // the call fails with left_ctx_short if the answer would depend on bytes before it)
  // out
  uint32_t rev_guess = 0;           // state assumed at own_hi
  uint32_t rev_left = 0;            // exact state at own_lo (what the left neighbour must assume)
  uint64_t exit_p = 0, exit_lm = 0; // iterator state leaving the shard
  uint64_t n_matches = 0;
  bool halo_overflow = false;
  bool left_ctx_short = false;
};

class DeviceBuf {
 public:
  ~DeviceBuf();
  void* ensure(size_t bytes);  // grow-only
  void* ptr = nullptr;
  size_t cap = 0;
};

class Regex {
 public:
  static Regex* compile(const std::vector<std::string>& patterns, const CompileOptions& opt, rb::Error* err);
  // The same patterns, options and pattern groups, compiled again (a second engine for another thread): a grouped
  // set compiles its planned groups directly and never repeats the determinization that failed.
  Regex* clone(rb::Error* err) const;
  ~Regex();

  size_t n_patterns() const { return patterns_.size(); }
  bool is_set() const { return is_set_; }
  // RegexSets in groups (DESIGN.md §2): first pattern index of each group; one entry (0) when one product
  // automaton covers the whole set, none for an empty set.
  std::vector<uint32_t> group_firsts() const {
    if (patterns_.empty()) return {};
    return groups_.empty() ? std::vector<uint32_t>{0} : group_first_;
  }
  bool grouped() const { return !groups_.empty(); }
  // Re-plan the groups with at most k patterns each (then split further by the table budget); 0 = automatic
  // (the product automaton when it fits).  Fails when a group does not compile; the plan is then unchanged.
  int set_group_patterns(uint32_t k);
  // Exclusive use of this object's device scratch for one call (the entry points lock mu_ themselves; the C ABI
  // uses these to find an idle engine when several threads share one rure*).
  bool try_acquire() { return mu_.try_lock(); }
  void acquire() { mu_.lock(); }
  void release() { mu_.unlock(); }
  const rb::Dfa* host_dfa(DfaKind k, rb::Error* err);  // builds lazily (also used by tests to inspect tables)

  // ---- single haystack, device-resident text --------------------------------
  // find_iter (re_trait.rs:197-220): writes up to cap {start,end} pairs to d_out
  // (device memory, may be null to count only); *total = number of matches.
  int find_all_device(const uint8_t* d_text, uint64_t n, uint64_t start, uint64_t* d_out, uint64_t cap, uint64_t* total);
  // the same over one shard of a sharded haystack; spans are buffer-relative
  int find_all_shard_device(const uint8_t* d_text, uint64_t n, ShardIO* io, uint64_t* d_out, uint64_t cap);
  // find_at (exec.rs:473-514)
  int find_at_device(const uint8_t* d_text, uint64_t n, uint64_t start, bool* found, uint64_t* s, uint64_t* e);
  // shortest_match_at / is_match_at (exec.rs:382-468); for sets: any pattern.
  int shortest_match_device(const uint8_t* d_text, uint64_t n, uint64_t start, bool* found, uint64_t* end);
  // RegexSet::matches (re_set.rs:184-213): masks = ceil(n_patterns/64) words (host).
  int set_matches_device(const uint8_t* d_text, uint64_t n, uint64_t start, bool* any, uint64_t* masks);

  // one shard of a forward search over a sharded haystack (see engine.cu)
  int forward_shard_device(const uint8_t* d_text, uint64_t n, uint64_t own_lo, uint64_t own_hi, bool is_first, bool is_last, uint32_t entry,
                           bool want_masks, bool* found, uint64_t* first_end, uint64_t* masks, uint32_t* entry_used, uint32_t* exit_state);

  // ---- bulk operations over the span list (re_bytes.rs:316-360 split/splitn, :476-535 replacen) ----
  // rep: replacement; expand = `$0`, `${0}`, `$$` as src/expand.rs (a reference to another group fails: captures
  // beyond group 0 are out of scope; NoExpand = expand false); limit 0 = all matches.  d_out may be null to size.
  int replace_device(const uint8_t* d_text, uint64_t n, const uint8_t* rep, uint64_t rep_len, bool expand, uint64_t limit,
                     uint8_t* d_out, uint64_t out_cap, uint64_t* out_len);
  int replace_host(const uint8_t* text, uint64_t n, const uint8_t* rep, uint64_t rep_len, bool expand, uint64_t limit,
                   uint8_t* out, uint64_t out_cap, uint64_t* out_len);
  // pieces as (start, end) pairs; has_limit/limit as splitn
  int split_device(const uint8_t* d_text, uint64_t n, bool has_limit, uint64_t limit, uint64_t* d_pieces, uint64_t cap, uint64_t* n_pieces);
  int split_host(const uint8_t* text, uint64_t n, bool has_limit, uint64_t limit, uint64_t* pieces, uint64_t cap, uint64_t* n_pieces);

  // ---- capture groups (exec.rs:527-590 read_captures_at, :861-875 captures_nfa_with_match) ----
  int n_groups() const { return n_groups_; }
  const std::vector<std::pair<std::string, int>>& group_names() const { return group_name_index_; }
  // slots of every match in d_spans: d_slots[m][2 * n_groups], kNone where a group did not take part
  int captures_device(const uint8_t* d_text, uint64_t n, const uint64_t* d_spans, uint64_t m, uint64_t* d_slots);
  // Regex::captures at `start` on a host haystack: slots[2 * n_groups]
  int captures_at_host(const uint8_t* text, uint64_t n, uint64_t start, bool* found, uint64_t* slots);
  // every match with its groups: slots[min(cap, *m)][2 * n_groups]
  int captures_all_host(const uint8_t* text, uint64_t n, uint64_t* slots, uint64_t cap, uint64_t* m);

  // ---- batched records, device-resident text + offsets[n_rec+1] --------------
  int is_match_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint32_t* d_bits);
  int find_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_spans, uint32_t* d_bits);
  int set_matches_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_masks);
  // find_iter per record (re_trait.rs:197-220, the record as the whole text): d_match_offsets[n_rec + 1] = exclusive
  // prefix sum of the per-record counts (always complete); record r's spans (record-relative) at
  // d_out[d_match_offsets[r] ..), at most cap stored (d_out may be null to count only); *total = all matches (host).
  int find_iter_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_match_offsets,
                             uint64_t* d_out, uint64_t cap, uint64_t* total);
  // Regex::captures per record: d_slots[n_rec][2 * n_groups] record-relative (kNone = no group); d_bits = ballot
  // words, bit r set when record r matches
  int captures_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_slots, uint32_t* d_bits);
  // replace_device per record (limit per record, 0 = all): record r's output is d_out[d_out_offsets[r] ..
  // d_out_offsets[r + 1]) (n_rec + 1 entries, always complete); at most out_cap bytes stored (d_out may be null to
  // size); *out_len = all output bytes (host)
  int replace_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, const uint8_t* rep, uint64_t rep_len, bool expand,
                           uint64_t limit, uint64_t* d_out_offsets, uint8_t* d_out, uint64_t out_cap, uint64_t* out_len);
  // split_device per record: record r's pieces (record-relative) at d_pieces[d_piece_offsets[r] ..), at most cap stored
  int split_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, bool has_limit, uint64_t limit, uint64_t* d_piece_offsets,
                         uint64_t* d_pieces, uint64_t cap, uint64_t* n_total);
  // captures_all_host per record: record r's matches at d_slots[d_match_offsets[r] ..][2 * n_groups], record-relative,
  // at most cap rows stored
  int captures_iter_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_match_offsets, uint64_t* d_slots,
                                 uint64_t cap, uint64_t* n_total);

  // ---- host-buffer wrappers (copies inside; the e2e path) ---------------------
  int find_all_host(const uint8_t* text, uint64_t n, uint64_t start, uint64_t* out, uint64_t cap, uint64_t* total);
  int find_at_host(const uint8_t* text, uint64_t n, uint64_t start, bool* found, uint64_t* s, uint64_t* e);
  int shortest_match_host(const uint8_t* text, uint64_t n, uint64_t start, bool* found, uint64_t* end);
  int set_matches_host(const uint8_t* text, uint64_t n, uint64_t start, bool* any, uint64_t* masks);
  int is_match_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint8_t* out_bits);
  int find_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* spans, uint8_t* out_bits);
  int set_matches_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* masks);
  int find_iter_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* match_offsets, uint64_t* out,
                           uint64_t cap, uint64_t* total);
  int captures_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* slots, uint8_t* out_bits);
  int replace_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, const uint8_t* rep, uint64_t rep_len, bool expand,
                         uint64_t limit, uint64_t* out_offsets, uint8_t* out, uint64_t out_cap, uint64_t* out_len);
  int split_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, bool has_limit, uint64_t limit, uint64_t* piece_offsets,
                       uint64_t* pieces, uint64_t cap, uint64_t* n_total);
  int captures_iter_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* match_offsets, uint64_t* slots,
                               uint64_t cap, uint64_t* n_total);

  // Run on a caller-owned CUDA stream (e.g. torch's current stream) instead of the private one.
  void set_stream(void* cuda_stream) { ext_stream_ = cuda_stream; use_ext_stream_ = true; }
  const std::string& last_error() const { return error_; }
  Tuning tuning;
  Stats stats;
  uint64_t min_len = 0, max_len = 0;  // match length range in bytes (max = kUnbounded)
  bool can_match_empty = false;
  bool has_looks = false;
  bool only_utf8 = false;
  // Candidate-start mode (DESIGN.md §2): a single pattern whose unanchored automata exceed the table budget is
  // searched from candidate starts with the anchored automaton (kinds 0 and 3); kinds 1, 2 and 4 are never built.
  bool candidate_mode() const { return !is_set_ && (unanchored_too_big_ || tuning.candidate_starts); }

 private:
  Regex() = default;
  struct DeviceDfa;
  int init_device();
  int d2h(void* dst, const void* src, size_t bytes);
  int ensure(DfaKind k, DeviceDfa** out);
  int fail(const std::string& msg);
  int check(int cuda_err, const char* what);
  struct ScanPlan { bool fast = false; uint32_t seg = 0, warm = 0; uint64_t n_seg = 0; };
  ScanPlan plan_scan(const uint8_t* d_text, uint64_t base, uint64_t limit, bool fast_table);
  // find_all_shard_device's path for one range (engine.cu): the start bitmap's scan plan, the path stats.path reports,
  // the chain walk's runner, chunk size, shared memory and kernels.  Also sets stats.path and stats.fused.
  struct WalkPlan;
  WalkPlan plan_walk(const uint8_t* d_text, const ShardIO& io, const DeviceDfa* fwd, const DeviceDfa* revall);
  int scan_starts(const uint8_t* d_text, uint64_t n, uint64_t base, uint64_t limit, ShardIO* io, const ScanPlan& plan,
                  const void* fused_walk);
  // Verify every segment's entry guess against its neighbour's exit (a.guess / a.fin, list in redo_) until none is
  // wrong: redo(n) launches the scan over the n listed segments; after max_redo_rounds rounds solve_entries.
  int settle_segments(const ScanArgs& a, bool reverse, const std::function<int(uint32_t)>& redo);
  int solve_entries(const ScanArgs& a, bool reverse);
  // State-map composition over the segments of g: K = the states below n_states that present_ marks (seeded by the
  // caller), closed under the per-segment maps; leaves in exact_ the entry state of every segment, the first one
  // in scan direction entered in the state at d_entry (device).
  int compose_entries(const ScanArgs& g, bool reverse, const uint16_t* d_entry);
  int resolve_long_run(const uint8_t* d_text, uint64_t n, uint64_t s, bool text_continues, uint64_t* e_out);
  // Bring the speculative chunk walks of *w into agreement with the sequential iterator (DESIGN.md §2): stitch_fast
  // when no match can be empty or look around, then general rounds until nothing changes.  rewalk(args, n) walks the
  // n chunks of args' dirty list again; after max_stitch_rounds rounds with re-walks, sequential(args) walks once from
  // args.seq_from.  Long runs a round requests are measured (resolve_long_run) and added to w->long_tab.
  // *grand_key: the general stitch's key of the whole range (device), null when it did not run.
  int stitch_chunks(WalkArgs* w, const std::function<int(const WalkArgs&, uint32_t)>& rewalk,
                    const std::function<int(const WalkArgs&)>& sequential, ChainKey** grand_key);
  int all_spans_device(const uint8_t* d_text, uint64_t n, uint64_t** d_spans, uint64_t* m);
  int ensure_capture_program();
  int launch_captures(const uint8_t* d_text, uint64_t n, const uint64_t* d_spans, uint64_t m, uint64_t* d_slots,
                      const uint64_t* rec_offsets, const uint32_t* rec_found, const uint64_t* rec_csr = nullptr, uint64_t n_rec = 0);
  // find_iter_batch_device; with grow (and d_out null) every span is stored in *grow, sized after the count pass
  int iter_batch(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_match_offsets, uint64_t* d_out, uint64_t cap,
                 uint64_t* total, DeviceBuf* grow);
  // exclusive prefix sum of in[0, n) into out (in == out allowed); *d_total = device address of the sum
  int prefix_sum(const uint64_t* in, uint64_t* out, uint64_t n, unsigned long long** d_total);
  // The fields every batched kernel takes (launch.h BatchArgs): views, text, offsets, n_rec, utf8; with the hot path
  // also the hot tables and the views' device copies.  Returns whether the hot path applies: hot tables for fwd and
  // rev (when given), 16-byte-aligned text, no force_generic, and max_per_sm > 0 (0: the caller has no hot kernel).
  // *smem: dynamic shared memory, the hot tables on the hot path, else fwd's class-indexed table (0: not staged).
  // *per_sm (hot path): blocks per SM, min(max_per_sm, 220 KiB / (*smem + reserve)), reserve = what a block is
  // budgeted beyond its tables.
  bool batch_args(BatchArgs* a, const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, DeviceDfa* fwd, DeviceDfa* rev,
                  size_t reserve, uint32_t max_per_sm, size_t* smem, uint32_t* per_sm);
  // text of every record of a host batch on the device (text_, boffsets_)
  int upload_batch(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, const uint8_t** d_text, uint64_t** d_offsets);
  int replace_prepare(const uint8_t* d_text, uint64_t n, const uint8_t* rep, uint64_t rep_len, bool expand, uint64_t limit, uint64_t* out_len);
  // the replacement template into rep_args_ / rep_lits_; *needs_groups = it refers to a group other than 0
  int replace_template(const uint8_t* rep, uint64_t rep_len, bool expand, bool* needs_groups);
  // prefix sums of the match and replacement lengths over m ordered spans of d_text[0, n) (slots: their groups, or null)
  int replace_sums(const uint8_t* d_text, uint64_t n, const uint64_t* spans, uint64_t m, const uint64_t* slots, uint64_t* out_len);
  int replace_emit(uint8_t* d_out, uint64_t out_cap);
  bool plan_prefilter();  // fills pf_words_ (launch.h PfArgs) when every match has one of <= 4 bytes at a fixed offset
  // ---- candidate-start mode ----
  int cand_args(void* out);  // launch.h CandArgs: byte sets of the first min(min_len, 4) offsets of a match
  // start bitmap (scan_rev format) of the candidates at positions (base, limit], plus position 0 when base == 0
  int cand_starts(const uint8_t* d_text, uint64_t n, uint64_t base, uint64_t limit, bool text_continues);
  int cand_shortest(const uint8_t* d_text, uint64_t n, uint64_t start, bool* found, uint64_t* end);
  // batched records from candidate starts: mode 0 is_match, 1 find, 2 / 3 find_iter count / write pass
  int cand_batch(int mode, const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint32_t* d_bits, uint64_t* d_spans,
                 uint64_t* d_match_offsets, uint64_t cap);
  int batch_route(bool* cand);  // batched find / find_iter: candidate starts, or kind 4 (switches to the mode when it is over budget)
  // words of forward_reduce's result: first match end + the pattern mask (at least kMaxMaskWords words)
  uint32_t result_words() const { return 1 + std::max<uint32_t>(4, (uint32_t)((patterns_.size() + 63) / 64)); }
  int forward_reduce(const uint8_t* d_text, uint64_t n, uint64_t start, bool want_masks, uint64_t* result_host, uint64_t end = ~0ull,
                     uint32_t entry = 0xFFFFFFFFu, uint32_t* exit_out = nullptr);
  int forward_range(const uint8_t* d_text, uint64_t n, uint64_t start, uint64_t limit, uint32_t entry, bool want_masks,
                    uint64_t* result_host, uint32_t* exit_state);
  int subset(const std::vector<uint32_t>& members, Regex** out);
  // Pattern groups: plan contiguous ranges of at most `chunk` patterns whose kind-2 automata fit the budget
  // (ranges over budget are halved); `plan` non-null compiles those ranges as given.
  static Regex* compile_impl(const std::vector<std::string>& patterns, const CompileOptions& opt, rb::Error* err,
                             const std::vector<uint32_t>* plan, uint32_t chunk);
  bool build_groups(const std::vector<uint32_t>* plan, uint32_t chunk, bool first_too_big, rb::Error* err);
  static Regex* compile_group(const std::vector<std::string>& all, uint32_t lo, uint32_t hi, const CompileOptions& opt, rb::Error* err);
  bool plan_range(uint32_t lo, uint32_t hi, bool known_too_big, std::vector<std::unique_ptr<Regex>>* out, std::vector<uint32_t>* firsts,
                  rb::Error* err);
  int set_matches_batch_grouped(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_masks);
  const uint8_t* upload_text(const uint8_t* text, uint64_t n, int* rc);
  int find_all_host_pipelined(const uint8_t* text, uint64_t n, uint8_t* d, uint64_t* d_out, uint64_t* out, uint64_t cap, uint64_t* total);
  int side_streams();  // creates copy_stream_ and back_stream_ on first use

  struct LazyUpload { const uint8_t* src; uint8_t* dst; uint64_t n, done; };  // host haystack uploaded wave by wave
  LazyUpload* lazy_ = nullptr;
  std::vector<std::string> patterns_;
  bool is_set_ = false;
  bool sparse_set_ = false;  // a narrowed RegexSet: none of its patterns matched in the first waves
  std::map<std::vector<uint32_t>, std::unique_ptr<Regex>> subsets_;
  std::vector<uint32_t> group_first_;                // grouped set: first pattern of each group
  std::vector<std::unique_ptr<Regex>> groups_;       // grouped set: one set-mode Regex per group (empty: one product automaton)
  bool product_fits_ = false;                        // the whole set's kind-2 automaton was determinized within budget
  DeviceBuf group_descs_;                            // launch.h GroupDesc per group (batched records)
  CompileOptions opt_;
  std::vector<rb::Expr> exprs_;
  std::unique_ptr<rb::Dfa> host_[kNumDfaKinds];
  bool unanchored_too_big_ = false;  // an unanchored automaton failed with DfaTooBig: candidate-start mode
  std::vector<uint8_t> cand_image_;  // launch.h CandArgs image (built on first use)
  DeviceDfa* dev_[kNumDfaKinds] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  std::string error_;
  std::recursive_mutex mu_;
  void* stream_ = nullptr;
  void* own_stream_ = nullptr;
  void* copy_stream_ = nullptr;  // host -> device pieces of a pipelined find_all
  void* back_stream_ = nullptr;  // device -> host spans of a pipelined find_all; the generic edge kernel of a forward scan
  void* ext_stream_ = nullptr;
  bool use_ext_stream_ = false;
  DeviceScalars* d_scalars_ = nullptr;  // counters, flags and reductions of the kernels (device)
  HostScalars* h_scalars_ = nullptr;    // pinned staging of the small copies to and from d_scalars_
  // ---- device scratch (grow-only), grouped by the calls that own it ----
  // whole-haystack scans (scan_starts, cand_starts, forward_range, settle_segments): start bitmap, segment entry
  // guesses and exits, redo list, per-segment forward results
  DeviceBuf bitmap_, guess_, fin_, redo_, seg_first_, seg_mask_;
  // state-map composition (solve_entries, compose_entries, resolve_long_run)
  DeviceBuf present_, kidx_, kstates_, maps_, comp_, bentry_, exact_;
  // chunk walk and stitch (find_all_shard_device, stitch_chunks): chain entries and exits, match counts and offsets,
  // dirty list, staged spans, stitch keys, resolved long runs
  DeviceBuf in_p_, in_lm_, out_p_, out_lm_, count_, offset_, dirty_, first_cand_, skip_, meta_, stage_, excl_, btot_, long_tab_;
  static constexpr uint32_t kMaxLongRuns = 256;
  DeviceBuf block_sums_;  // prefix_sum (any caller)
  // replace / split over one haystack: all spans, match lengths and the prefix sums of the match and replacement
  // lengths, template literals
  DeviceBuf spans_all_, lens_, lens_before_, reps_before_, lits_;
  uint64_t rep_totals_[2] = {0, 0};  // matched bytes, replacement bytes of the pending replace call
  std::vector<uint8_t> rep_args_, rep_lits_;  // launch.h ReplaceArgs image + literal bytes of the pending replace call
  int n_groups_ = 1;                      // capture groups incl. group 0
  std::vector<std::string> group_names_;  // names of the named groups
  std::vector<std::pair<std::string, int>> group_name_index_;  // (name, group index)
  DeviceBuf cap_insts_, cap_scratch_, cap_slots_, cap_span_;
  uint32_t cap_n_insts_ = 0, cap_start_ = 0;  // capture program on the device (0 = not uploaded yet)
  bool cap_anchored_ = false;
  // batched records (never shared with the whole-haystack calls, which the per-record captures_iter redo runs in
  // between): match CSR and spans, kept CSR and spans, slots, divergence flags and list; the record offsets of
  // every batched host wrapper (boffsets_) and the CSR and items of the find_iter / replace / split / captures_iter
  // host wrappers (bres_off_, bres_)
  DeviceBuf bmoff_, bspans_, bkoff_, bkspans_, bslots_, bflags_, blist_, boffsets_, bres_off_, bres_;
  // host wrappers: the haystack, spans (also find_at_device's one span), split pieces, replace output, batched match
  // bits and set masks
  DeviceBuf text_, out_, pieces_, rep_out_, bits_, masks_;
  void* timing_events_[3] = {nullptr, nullptr, nullptr};
  void *fork_event_ = nullptr, *join_event_ = nullptr;  // forward scans: the generic edge kernel runs beside the fast one
  int pf_state_ = 0;               // 0 = not decided yet, 1 = prefilter applies, -1 = it does not
  uint32_t pf_freq_ = 0;           // estimated frequency of the scanned bytes, parts per 65536
  std::vector<uint32_t> pf_words_; // PfArgs image (engine.cu)
};

uint64_t kernel_launches();  // total kernels launched by this library in this process
int device_sm_count();

}  // namespace rbgpu
