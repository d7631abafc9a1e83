// Host orchestration of the search kernels.  See engine.h.
#include "engine.h"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <unordered_map>

#include "launch.h"

namespace rbgpu {

// cuTensorMapEncodeTiled through the runtime (the library links cudart statically, not libcuda).
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// 2-D view of `rows` consecutive segments of `seg` bytes from `base` for the fast scan kernels' tiled TMA loads
// (rows = segments, cols = bytes); one box = the 64-byte group of all 32 lanes' segments.
static bool encode_segments(CUtensorMap* tmap, const uint8_t* base, uint32_t seg, uint64_t rows) {
  if (!encode_tiled()) return false;
  cuuint64_t dims[2] = {seg, rows};
  cuuint64_t strides[1] = {seg};
  cuuint32_t box[2] = {64, 32};
  cuuint32_t estr[2] = {1, 1};
  return encode_tiled()(tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static std::atomic<uint64_t> g_launches{0};
uint64_t kernel_launches() { return g_launches.load(); }

int device_sm_count() {
  static int sms = -1;
  if (sms < 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 0;
  }
  return sms;
}

DeviceBuf::~DeviceBuf() { if (ptr) cudaFree(ptr); }
void* DeviceBuf::ensure(size_t bytes) {
  if (bytes <= cap) return ptr;
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
  size_t want = std::max<size_t>(bytes, 256);
  if (cudaMalloc(&ptr, want) != cudaSuccess) { ptr = nullptr; return nullptr; }
  cap = want;
  return ptr;
}

// Hot tables of up to this many rows (288 bytes per row, one-byte successor ids) are
// staged in shared memory by the fast kernels.
static constexpr uint32_t kFastStates = 200;
static size_t hot_bytes(uint32_t rows) { return ((size_t)rows * RB_HOT_ROW + 255) / 256 * 256; }  // kernels.cu hot_table_bytes
// scan_rev_fast's reverse table with signed row ids (kernels.cu hot_signed_bytes): match rows and the others are rounded apart
static size_t hot_bytes_signed(const HotView& h) { return hot_bytes(h.n - h.match_lo) + hot_bytes(h.match_lo); }
static bool hot_signed_ok(const HotView& h) { return h.n != 0 && h.match_lo <= 128 && h.n - h.match_lo <= 128; }

struct Regex::DeviceDfa {
  DfaView view;
  void* trans = nullptr;
  void* classes = nullptr;
  void* masks = nullptr;
  // byte-indexed expansion over the hot states for the fast kernels (kernels.cuh HotView);
  // hot.n == 0 when even the ASCII-reachable part has more than kFastStates states
  void* next256 = nullptr;
  void* eof = nullptr;
  void* hot2full = nullptr;
  void* full2hot = nullptr;
  void* view_dev = nullptr;  // copy of `view` in global memory (cold fallbacks take a pointer)
  HotView hot{};
  ~DeviceDfa() {
    cudaFree(trans); cudaFree(classes); cudaFree(masks); cudaFree(next256); cudaFree(eof);
    cudaFree(hot2full); cudaFree(full2hot); cudaFree(view_dev);
  }
};

// The scalars kernels count, flag or reduce into (one per object, allocated by init_device).  No two fields share
// bytes; where one copy or memset covers several fields, an assert below keeps them together.
struct DeviceScalars {
  // settle_segments: [0] segments to redo.  Stitch (launch.h stitch_fast / stitch_resolve): [0] chunks to walk
  // again, [1] changed decisions, [2] the general loop is needed, [3] smallest chunk index to walk again
  uint32_t list[4];
  unsigned long long long_req;   // stitch: smallest start of a run longer than kExactRunCap (kNone = none)
  unsigned long long long_best;  // resolve_long_run: last match end + 1 in the window (0 = none)
  uint32_t long_alive;           // resolve_long_run: the run is still alive at the window's end
  uint32_t n_new;                // compose_entries: states closure_check added to K
  uint32_t err_flag;             // walks: a match runs past the end of a shard's halo
  uint32_t floor_flag;           // walks: a reverse-on-slice scan reaches the left end of the buffer
  uint32_t first_deferred;       // stitch: entries_local's leftmost deferred chunk
  uint16_t long_entry;           // resolve_long_run: the automaton's state at the run's start
  uint8_t flag0;                 // start bitmaps: a match starts at position 0
  unsigned long long task_counter;  // batch_refill: next task to hand out
  unsigned long long cand_best;     // cand_shortest: earliest match end
  uint32_t cand_overflow;           // cand_shortest in a stream's window: a run reached the window's end undecided
  unsigned long long fwd_result[1 + kMaxMaskWords];  // forward_range: first match end, OR of the pattern masks
};

// Pinned host side of the small copies (init_device).  A field staged for an async host-to-device copy is not
// written again before the stream synchronises.
struct HostScalars {
  uint32_t list[4];              // a stitch round: DeviceScalars::list and long_req in one copy
  unsigned long long long_req;
  uint32_t n_redo;               // settle_segments
  uint32_t err_flag, floor_flag; // find_all: DeviceScalars::err_flag and floor_flag in one copy
  uint64_t n_matches;            // find_all
  uint64_t exit[2];              // find_all: iterator state leaving the range (ChainKey, or out_p / out_lm of the last chunk)
  uint64_t iter_total;           // iter_batch: matches of all records
  uint64_t fwd_result[1 + kMaxMaskWords];  // forward_range: the initial result (staged), then the reduced one
  uint16_t fwd_exit;             // forward_range: exit state
  uint16_t rev_guess, rev_left;  // scan_starts, a shard: reverse-scan state assumed at own_hi, exact state at own_lo
  uint16_t seed_state;           // scan_starts, a shard: the exact state at own_hi (staged) ...
  uint32_t seed_seg, seed_count; // ... for one redo round of the top segment (staged)
};

// b directly follows a: one copy or memset covers both
#define RB_FOLLOWS(S, a, b) static_assert(offsetof(S, b) == offsetof(S, a) + sizeof(S::a), #S ": " #b " must follow " #a)
RB_FOLLOWS(DeviceScalars, list, long_req);
RB_FOLLOWS(HostScalars, list, long_req);
RB_FOLLOWS(DeviceScalars, long_best, long_alive);
RB_FOLLOWS(DeviceScalars, err_flag, floor_flag);
RB_FOLLOWS(HostScalars, err_flag, floor_flag);
#undef RB_FOLLOWS
static_assert(offsetof(DeviceScalars, first_deferred) == offsetof(DeviceScalars, list) + 12 * sizeof(uint32_t),
              "stitch_resolve reads the leftmost deferred chunk as counters[12]");

// ------------------------------------------------------------------ compile --
Regex* Regex::compile(const std::vector<std::string>& patterns, const CompileOptions& opt, rb::Error* err) {
  return compile_impl(patterns, opt, err, nullptr, 0);
}

Regex* Regex::clone(rb::Error* err) const {
  const std::vector<uint32_t> one{0};
  return compile_impl(patterns_, opt_, err, groups_.empty() ? &one : &group_first_, 0);
}

// plan: null = automatic (the product automaton of a set of <= 256 patterns when it fits, else pattern groups);
// {0} = one product automaton or its error; more entries = exactly these groups.  chunk: groups of at most this many
// patterns before the budget splits them (set_group_patterns), 0 = automatic.
Regex* Regex::compile_impl(const std::vector<std::string>& patterns, const CompileOptions& opt, rb::Error* err,
                           const std::vector<uint32_t>* plan, uint32_t chunk) {
  std::unique_ptr<Regex> re(new Regex());
  re->patterns_ = patterns;
  re->opt_ = opt;
  re->only_utf8 = opt.only_utf8;
  re->is_set_ = opt.as_set || patterns.size() != 1;
  rb::Flags f;
  f.casei = opt.flags & 1; f.multi = opt.flags & 2; f.dotnl = opt.flags & 4; f.swap_greed = opt.flags & 8;
  f.ignore_space = opt.flags & 16; f.unicode = opt.flags & 32;
  f.allow_bytes = !opt.only_utf8;  // exec.rs:224-225
  re->exprs_.resize(patterns.size());
  re->min_len = rb::kUnbounded;
  re->max_len = 0;
  for (size_t i = 0; i < patterns.size(); i++) {
    if (!rb::parse(patterns[i], f, 200, &re->exprs_[i], err)) return nullptr;
    uint64_t mn, mx;
    rb::expr_len_range(re->exprs_[i], &mn, &mx);
    re->min_len = std::min(re->min_len, mn);
    re->max_len = std::max(re->max_len, mx);
  }
  if (patterns.size() == 1) {  // capture groups of the pattern (only their existence matters: replacement templates)
    std::vector<const rb::Expr*> stack{&re->exprs_[0]};
    while (!stack.empty()) {
      const rb::Expr* x = stack.back();
      stack.pop_back();
      if (x->kind == rb::EK::Group && x->cap > 0) {
        re->n_groups_ = std::max(re->n_groups_, x->cap + 1);
        if (!x->name.empty()) { re->group_names_.push_back(x->name); re->group_name_index_.emplace_back(x->name, x->cap); }
      }
      for (const rb::Expr& c : x->es) stack.push_back(&c);
    }
  }
  if (patterns.empty()) { re->min_len = 0; return re.release(); }
  re->can_match_empty = re->min_len == 0;
  // Validate eagerly what the reference validates at build time (program size)
  // plus the two explicit errors of this backend (Unicode \b, table budget).
  rb::Program probe;
  rb::CompileOptions co;
  co.only_utf8 = opt.only_utf8;
  co.size_limit = opt.size_limit;
  if (!rb::compile(re->exprs_, co, &probe, err)) return nullptr;
  re->has_looks = probe.has_looks;
  if (probe.has_unicode_word_boundary) {
    err->kind = rb::Error::UnicodeWordBoundary;
    err->msg = "Unicode word boundaries (\\b, \\B) are not supported by the B200 DFA backend; use (?-u:\\b).";
    return nullptr;
  }
  // Determinize the tables every object needs so budget errors surface at compile time.
  if (re->is_set_) {
    // Set semantics need the all-match automaton of every pattern, or (DESIGN.md §2, RegexSets in groups) the
    // automata of contiguous pattern ranges: matches[i] only says that pattern i matches somewhere, so the OR of
    // the groups' masks is the same answer.  A group holds at most 64 * kMaxMaskWords patterns.
    if (plan && plan->size() > 1) return re->build_groups(plan, 0, false, err) ? re.release() : nullptr;
    const bool one_table = plan != nullptr;
    if (one_table || (chunk == 0 && patterns.size() <= 64 * kMaxMaskWords)) {
      if (re->host_dfa(kFwdUnanchoredAll, err)) { re->product_fits_ = true; return re.release(); }
      if (one_table || err->kind != rb::Error::DfaTooBig || patterns.size() == 1) return nullptr;
    }
    *err = rb::Error();
    // a set of <= 256 patterns lands here after its product automaton failed: that range is split at once
    return re->build_groups(nullptr, chunk ? chunk : 64 * kMaxMaskWords, patterns.size() <= 64 * kMaxMaskWords && chunk == 0, err)
               ? re.release() : nullptr;
  }
  // A single pattern: the anchored automaton first (cheap).  When it fits but an unanchored one does not (it tracks
  // every earlier start that may still begin a match: `error.{0,100}timeout` has 2^100 such subsets), the object
  // searches from candidate starts with kinds 0 and 3 (DESIGN.md §2).  Only one over-budget unanchored
  // determinization is paid for.  When kind 0 or kind 3 is over budget as well, the error is the one an eager
  // kind 2, 0, 1 sequence reports.
  if (!re->host_dfa(kFwdAnchoredLF, err)) {
    rb::Error e2;
    if (!re->host_dfa(kFwdUnanchoredAll, &e2)) *err = e2;
    return nullptr;
  }
  for (DfaKind k : {kFwdUnanchoredAll, kRevUnanchoredAll}) {
    if (re->host_dfa(k, err)) continue;
    if (err->kind != rb::Error::DfaTooBig) return nullptr;
    rb::Error e3;
    if (!re->host_dfa(kRevAnchoredLongest, &e3)) return nullptr;  // *err: the unanchored automaton's error
    re->unanchored_too_big_ = true;
    for (DfaKind u : {kRevUnanchoredAll, kFwdUnanchoredAll, kFwdUnanchoredLF}) re->host_[u].reset();
    *err = rb::Error();
    break;
  }
  return re.release();
}

Regex::~Regex() {
  for (auto*& d : dev_) { delete d; d = nullptr; }
  if (h_scalars_) cudaFreeHost(h_scalars_);
  if (d_scalars_) cudaFree(d_scalars_);
  for (void* e : timing_events_) if (e) cudaEventDestroy((cudaEvent_t)e);
  if (fork_event_) cudaEventDestroy((cudaEvent_t)fork_event_);
  if (join_event_) cudaEventDestroy((cudaEvent_t)join_event_);
  if (copy_stream_) cudaStreamDestroy((cudaStream_t)copy_stream_);
  if (back_stream_) cudaStreamDestroy((cudaStream_t)back_stream_);
  if (own_stream_) cudaStreamDestroy((cudaStream_t)own_stream_);
}

const rb::Dfa* Regex::host_dfa(DfaKind k, rb::Error* err) {
  if (host_[k]) return host_[k].get();
  if (patterns_.empty()) {  // an empty RegexSet matches nothing and has no automaton
    err->kind = rb::Error::Syntax;
    err->msg = "an empty pattern set has no automaton";
    return nullptr;
  }
  if (k == kFwdUnanchoredAll && !groups_.empty()) {
    std::string ranges;
    for (size_t g = 0; g < groups_.size(); g++)
      ranges += (g ? ", [" : "[") + std::to_string(group_first_[g]) + ", " +
                std::to_string(g + 1 < groups_.size() ? group_first_[g + 1] : patterns_.size()) + ")";
    err->kind = rb::Error::DfaTooBig;
    err->msg = "this RegexSet is searched in " + std::to_string(groups_.size()) + " pattern groups (" + ranges +
               "), each with its own automaton; there is no product automaton of the whole set";
    return nullptr;
  }
  if (unanchored_too_big_ && k != kFwdAnchoredLF && k != kRevAnchoredLongest) {
    err->kind = rb::Error::DfaTooBig;
    err->msg = "the unanchored automata of this pattern exceed the DFA table budget: it is searched from candidate starts "
               "with the anchored automata (kinds 0 and 3) only";
    return nullptr;
  }
  rb::CompileOptions co;
  co.only_utf8 = opt_.only_utf8;
  co.size_limit = opt_.size_limit;
  rb::DfaOptions dopt;
  dopt.max_table_bytes = opt_.dfa_size_limit * 16;
  switch (k) {
    case kFwdAnchoredLF: co.reverse = false; co.unanchored_prefix = false; dopt.anchored = true; dopt.leftmost_first = true; break;
    case kRevUnanchoredAll: co.reverse = true; co.unanchored_prefix = true; dopt.anchored = false; dopt.leftmost_first = false; break;
    case kFwdUnanchoredAll: co.reverse = false; co.unanchored_prefix = true; dopt.anchored = false; dopt.leftmost_first = false; break;
    case kRevAnchoredLongest: co.reverse = true; co.unanchored_prefix = false; dopt.anchored = true; dopt.leftmost_first = false; break;
    case kFwdUnanchoredLF: co.reverse = false; co.unanchored_prefix = true; dopt.anchored = false; dopt.leftmost_first = true; break;
    default: return nullptr;
  }
  if (is_set_ || patterns_.size() != 1) dopt.leftmost_first = false;  // dfa.rs:1557-1559
  rb::Program prog;
  if (!rb::compile(exprs_, co, &prog, err)) return nullptr;
  std::unique_ptr<rb::Dfa> d(new rb::Dfa());
  if (!rb::determinize(prog, dopt, d.get(), err)) return nullptr;
  host_[k] = std::move(d);
  return host_[k].get();
}

int Regex::fail(const std::string& msg) {
  error_ = msg;
  return -1;
}
int Regex::check(int e, const char* what) {
  if (e == cudaSuccess) return 0;
  return fail(std::string("CUDA error in ") + what + ": " + cudaGetErrorString((cudaError_t)e));
}
#define RB_CUDA(call)                                   \
  do {                                                  \
    int rc__ = check((int)(call), #call);               \
    if (rc__) return rc__;                              \
  } while (0)
#define RB_LAUNCH_CHECK(name)                           \
  do {                                                  \
    g_launches++;                                       \
    int rc__ = check((int)cudaGetLastError(), name);    \
    if (rc__) return rc__;                              \
  } while (0)

// Stream, device and pinned scalars and timing events of this object.  Every copy and kernel of the
// library is issued on stream_ (or on the two pipeline streams, ordered by events).  The
// library's own stream is a BLOCKING stream: it is ordered with the legacy default stream,
// which is where a caller that never heard of streams (or torch's default stream) produced the
// device buffers it hands to the *_device entry points -- a non-blocking stream raced with
// `torch.zeros(...)` of the output buffer in the tests.  Callers on another stream pass it
// with rure_b200_set_stream.
int Regex::init_device() {
  if (!h_scalars_) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
      return fail("no CUDA device available: regex_b200 has no CPU matching path");
    cudaStream_t s;
    RB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamDefault));
    own_stream_ = s;
    RB_CUDA(cudaMalloc(&d_scalars_, sizeof(DeviceScalars)));
    RB_CUDA(cudaMallocHost(&h_scalars_, sizeof(HostScalars)));
    for (void*& e : timing_events_) {
      cudaEvent_t ev;
      RB_CUDA(cudaEventCreate(&ev));
      e = ev;
    }
  }
  stream_ = use_ext_stream_ ? ext_stream_ : own_stream_;
  return 0;
}

int Regex::ensure(DfaKind k, DeviceDfa** out) {
  if (int rc = init_device()) return rc;
  if (dev_[k]) { *out = dev_[k]; return 0; }
  cudaStream_t up = (cudaStream_t)stream_;
  rb::Error err;
  const rb::Dfa* h = host_dfa(k, &err);
  if (!h) return fail(err.msg);
  std::unique_ptr<DeviceDfa> d(new DeviceDfa());
  const size_t tb = h->trans.size() * sizeof(uint16_t);
  RB_CUDA(cudaMalloc(&d->trans, std::max<size_t>(tb, 16)));
  RB_CUDA(cudaMalloc(&d->classes, 256));
  RB_CUDA(cudaMalloc(&d->masks, std::max<size_t>(h->masks.size() * 8, 16)));
  RB_CUDA(cudaMemcpyAsync(d->trans, h->trans.data(), tb, cudaMemcpyHostToDevice, up));
  RB_CUDA(cudaMemcpyAsync(d->classes, h->classes, 256, cudaMemcpyHostToDevice, up));
  RB_CUDA(cudaMemcpyAsync(d->masks, h->masks.data(), h->masks.size() * 8, cudaMemcpyHostToDevice, up));
  DfaView& v = d->view;
  v.trans = (const uint16_t*)d->trans;
  v.classes = (const uint8_t*)d->classes;
  v.masks = (const uint64_t*)d->masks;
  v.n_states = h->n_states;
  v.stride = h->n_classes;
  v.match_lo = h->match_lo;
  v.mask_words = h->mask_words;
  v.table_bytes = (uint32_t)tb;
  std::memcpy(v.start, h->start, sizeof v.start);
  v.uniform_start = h->uniform_start;
  // Hot set: every state when they all fit, else the closure of the start states under
  // ASCII bytes (what an ASCII haystack can reach).  Row 1 is the trap.
  {
    std::vector<uint8_t> is_hot(h->n_states, 0);
    {
      std::vector<uint16_t> stack;
      auto push = [&](uint16_t s) { if (!is_hot[s]) { is_hot[s] = 1; stack.push_back(s); } };
      push(0);
      for (uint16_t s : h->start) push(s);
      while (!stack.empty()) {
        const uint16_t s = stack.back();
        stack.pop_back();
        for (int b = 0; b < 128; b++) push(h->next(s, (uint8_t)b));
      }
    }
    // All states when they fit -- unless the ASCII closure is a small part of the automaton: Unicode `\d`
    // in `(\d{4})-(\d{2})-(\d{2})` makes 183 states of which 15 are reachable on ASCII, and a 51 KB table
    // costs a block per SM and most of the L1 where 4 KB will do (non-ASCII bytes take the trap row).
    const size_t n_closure = (size_t)std::count(is_hot.begin(), is_hot.end(), 1);
    if (h->n_states + 1 <= kFastStates && n_closure * 4 > h->n_states) std::fill(is_hot.begin(), is_hot.end(), 1);
    const size_t n_hot = (size_t)std::count(is_hot.begin(), is_hot.end(), 1) + 1;
    if (n_hot <= kFastStates) {
      std::vector<uint16_t> full2hot(h->n_states, 0xFFFF), hot2full;
      hot2full.push_back(0);       // dead
      hot2full.push_back(0xFFFF);  // trap
      full2hot[0] = 0;
      for (uint32_t s = 1; s < h->n_states; s++)  // full ids are already ordered non-match < match
        if (is_hot[s]) { full2hot[s] = (uint16_t)hot2full.size(); hot2full.push_back((uint16_t)s); }
      uint32_t hot_match_lo = (uint32_t)hot2full.size();
      for (uint32_t i = 2; i < hot2full.size(); i++)
        if (hot2full[i] >= h->match_lo) { hot_match_lo = i; break; }
      std::vector<uint16_t> n256(hot2full.size() * 256), eof(hot2full.size(), 0);
      for (uint32_t r = 0; r < hot2full.size(); r++) {
        for (int b = 0; b < 256; b++) {
          uint16_t to = 1;  // trap row: absorbing
          if (r != 1) {
            const uint16_t t = full2hot[h->next(hot2full[r], (uint8_t)b)];
            to = t == 0xFFFF ? 1 : t;
          }
          n256[(size_t)r * 256 + b] = to;
        }
        if (r != 1) eof[r] = h->next_eof(hot2full[r]);
      }
      RB_CUDA(cudaMalloc(&d->next256, n256.size() * 2));
      RB_CUDA(cudaMalloc(&d->eof, eof.size() * 2));
      RB_CUDA(cudaMalloc(&d->hot2full, hot2full.size() * 2));
      RB_CUDA(cudaMalloc(&d->full2hot, full2hot.size() * 2));
      RB_CUDA(cudaMemcpyAsync(d->next256, n256.data(), n256.size() * 2, cudaMemcpyHostToDevice, up));
      RB_CUDA(cudaMemcpyAsync(d->eof, eof.data(), eof.size() * 2, cudaMemcpyHostToDevice, up));
      RB_CUDA(cudaMemcpyAsync(d->hot2full, hot2full.data(), hot2full.size() * 2, cudaMemcpyHostToDevice, up));
      RB_CUDA(cudaMemcpyAsync(d->full2hot, full2hot.data(), full2hot.size() * 2, cudaMemcpyHostToDevice, up));
      RB_CUDA(cudaStreamSynchronize(up));  // the host vectors above die with this scope
      d->hot.next256 = (const uint16_t*)d->next256;
      d->hot.eof = (const uint16_t*)d->eof;
      d->hot.hot2full = (const uint16_t*)d->hot2full;
      d->hot.full2hot = (const uint16_t*)d->full2hot;
      d->hot.n = (uint32_t)hot2full.size();
      d->hot.match_lo = hot_match_lo;
      d->hot.start = full2hot[h->start[32]];
    }
  }
  RB_CUDA(cudaMalloc(&d->view_dev, sizeof(DfaView)));
  RB_CUDA(cudaMemcpyAsync(d->view_dev, &d->view, sizeof(DfaView), cudaMemcpyHostToDevice, up));
  RB_CUDA(cudaStreamSynchronize(up));
  dev_[k] = d.release();
  *out = dev_[k];
  return 0;
}

// Shared-memory staging decision: table + class map must fit the opt-in limit.
static size_t smem_for(const DfaView& v) {
  size_t need = ((size_t)v.table_bytes + 15) / 16 * 16 + 256;
  return need <= 200 * 1024 ? need : 0;
}
// Opt a kernel in to `bytes` of dynamic shared memory.  The attribute belongs to the function, not to the
// caller: it is only ever RAISED (per-kernel maximum under a lock) -- two regex objects with different table
// sizes searching from two threads would otherwise lower it under each other's launches ("invalid argument").
// min_bytes: kernels with static shared memory on top pass 48 KB so that the sum may exceed the default limit.
template <typename K>
static cudaError_t allow_smem(K kernel, size_t bytes, size_t min_bytes = 0) {
  bytes = std::max(bytes, min_bytes);
  if (bytes <= 48 * 1024 && min_bytes == 0) return cudaSuccess;
  static std::mutex mu;
  static std::unordered_map<const void*, size_t> granted;
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = granted[(const void*)kernel];
  if (bytes <= have) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) have = bytes;
  return e;
}
static uint32_t grid_for(uint64_t threads_needed, uint32_t block, uint32_t blocks_per_sm) {
  uint64_t blocks = (threads_needed + block - 1) / block;
  uint64_t cap = (uint64_t)std::max(1, device_sm_count()) * blocks_per_sm;
  return (uint32_t)std::max<uint64_t>(1, std::min(blocks, cap));
}

// The most dynamic shared memory a block can opt in to on sm_100 (allow_smem).
static constexpr size_t kMaxDynamicSmem = 227 * 1024;
static size_t fast_scan_smem(size_t table_bytes) {
  return table_bytes + 1024 + (1024 / 32) * (2 * 2048 + 64);  // kernels.cu kBoxStages, kRingBarBytes  // kernels.cu: tables, 512-aligned rings, mbarriers
}

static uint32_t pick_warm(const Regex& re) {
  if (re.tuning.warm) return (re.tuning.warm + 15) / 16 * 16;
  if (re.max_len != rb::kUnbounded) return (uint32_t)std::min<uint64_t>((std::max<uint64_t>(re.max_len, 1) + 15) / 16 * 16, 4096);
  return 128;
}

// ---------------------------------------------------------- literal prefilter --
// Estimated byte frequencies, parts per 65536 (tools/gen_byte_freq.py).
static const uint16_t kByteFreq[256] = {
#include "byte_freq.inc"
};
// A pattern qualifies when every match must have one of at most four bytes of small total
// estimated frequency at some fixed offset o < min_len (the reference scans for its rarest
// literal byte, src/literals.rs:466-489; here the bytes come from the automaton, so character
// classes and alternations qualify as well: `Sher[a-z]+|Hol[a-z]+` scans for S and H).
// Measured on the B200 (profiles/r02_prefilter.md): the word-wide byte tests cost ~2.3
// instructions per haystack byte for two byte values, and every hit costs a queue push plus its
// share of a verification round, against 5 instructions per byte for the shared-memory DFA scan.
// `Holmes|Watson` over the C2 corpus (an H or W every 238 bytes, a match every 1.1 KB) runs at
// 1.33 TB/s here and at 2.93 TB/s on the fused DFA path, so the automatic choice is conservative:
static constexpr uint32_t kPrefilterMaxFreq = 600;   // structural limit (tuning.prefilter == 2): ~0.9 % of the bytes
static constexpr uint32_t kPrefilterAutoFreq = 80;   // automatic (tuning.prefilter == 1): ~0.12 %, i.e. one rare byte
static constexpr uint32_t kPrefilterState = 0xFFFEu; // what a prefilter or candidate-start shard reports as its boundary states

// allowed[d][b] = 1 when some start state of the anchored automaton d survives d + 1 steps with byte b as the last one
// (every match of at least `depth` bytes has such a byte at offset d).  Start states: all of them unless uniform.
static std::vector<std::vector<uint8_t>> start_byte_sets(const rb::Dfa& d, uint32_t depth) {
  std::vector<std::vector<uint8_t>> allowed(depth, std::vector<uint8_t>(256, 0));
  std::vector<uint8_t> reach(d.n_states, 0), next(d.n_states, 0);
  if (d.uniform_start) reach[d.start[32]] = 1;
  else for (uint16_t s : d.start) reach[s] = 1;
  reach[0] = 0;
  for (uint32_t dep = 0; dep < depth; dep++) {
    std::fill(next.begin(), next.end(), 0);
    for (uint32_t st = 1; st < d.n_states; st++) {
      if (!reach[st]) continue;
      for (int b = 0; b < 256; b++) {
        const uint16_t t = d.next((uint16_t)st, (uint8_t)b);
        if (t) { allowed[dep][b] = 1; next[t] = 1; }
      }
    }
    reach.swap(next);
  }
  return allowed;
}

bool Regex::plan_prefilter() {
  if (pf_state_) return pf_state_ > 0;
  pf_state_ = -1;
  if (is_set_ || has_looks || min_len == 0 || patterns_.size() != 1) return false;
  rb::Error err;
  const rb::Dfa* d = host_dfa(kFwdAnchoredLF, &err);
  if (!d || !d->uniform_start) return false;
  const uint32_t depth = (uint32_t)std::min<uint64_t>(min_len, 8);
  const std::vector<std::vector<uint8_t>> allowed = start_byte_sets(*d, depth);
  uint32_t best_o = 0, best_f = ~0u;
  for (uint32_t o = 0; o < depth; o++) {
    uint32_t cnt = 0, f = 0;
    for (int b = 0; b < 256; b++) if (allowed[o][b]) { cnt++; f += kByteFreq[b]; }
    if (cnt >= 1 && cnt <= 4 && f < best_f) { best_f = f; best_o = o; }
  }
  if (best_f > kPrefilterMaxFreq) return false;
  PfArgs a{};
  a.o = best_o;
  for (int b = 0; b < 256; b++) if (allowed[best_o][b]) a.bcast[a.n_bytes++] = 0x01010101u * (uint32_t)b;
  a.n_sets = std::min<uint32_t>(depth, 4);
  for (uint32_t dep = 0; dep < a.n_sets; dep++)
    for (int b = 0; b < 256; b++) if (allowed[dep][b]) a.sets[dep][b >> 5] |= 1u << (b & 31);
  pf_words_.resize(sizeof(PfArgs) / 4);
  std::memcpy(pf_words_.data(), &a, sizeof a);
  pf_freq_ = best_f;
  pf_state_ = 1;
  return true;
}

// ---------------------------------------------------------- candidate starts --
// Candidate-start mode (DESIGN.md §2).  find_at(p) = (s*, A(s*)) with s* the first position >= p at which the
// anchored automaton A finds a match; that holds for any superset of the match starts, so kind 0 (and kind 3 for
// the reverse-on-slice rule) answers every single-pattern call.  The candidates: positions whose first
// D = min(min_len, 4) bytes lie in the byte sets of start_byte_sets; every position when min_len == 0.
int Regex::cand_args(void* out) {
  if (cand_image_.empty()) {
    rb::Error err;
    const rb::Dfa* d = host_dfa(kFwdAnchoredLF, &err);
    if (!d) return fail(err.msg);
    CandArgs c{};
    c.depth = (uint32_t)std::min<uint64_t>(min_len, 4);
    const std::vector<std::vector<uint8_t>> allowed = start_byte_sets(*d, c.depth);
    for (uint32_t dep = 0; dep < c.depth; dep++)
      for (int b = 0; b < 256; b++) if (allowed[dep][b]) c.mask[b] |= (uint8_t)(1u << dep);
    c.utf8_boundaries = only_utf8 && can_match_empty;  // as scan_starts: the reverse scan drops those starts too
    c.slice_rule = has_looks;
    cand_image_.resize(sizeof c);
    std::memcpy(cand_image_.data(), &c, sizeof c);
  }
  std::memcpy(out, cand_image_.data(), sizeof(CandArgs));
  return 0;
}

int Regex::cand_starts(const uint8_t* d_text, uint64_t n, uint64_t base, uint64_t limit, bool text_continues) {
  CandArgs c;
  if (int rc = cand_args(&c)) return rc;
  uint64_t* bm = (uint64_t*)bitmap_.ensure(((n >> 6) + 2) * 8);
  if (!bm) return fail("out of device memory (bitmap)");
  const uint64_t words = std::max<uint64_t>(1, ((limit + 63) >> 6) - (base >> 6));
  cand_bitmap<<<grid_for(words, 256, 8), 256, 0, (cudaStream_t)stream_>>>(d_text, n, base, limit, text_continues ? 1 : 0, c, bm,
                                                                        &d_scalars_->flag0);
  RB_LAUNCH_CHECK("cand_bitmap");
  return 0;
}

// shortest_match / is_match: min over the candidates s >= start of the first match state the anchored automaton
// enters from s, in the waves of forward_reduce (64 MiB, x16 each); a wave is the last one once the best end lies
// at or before the next wave's first candidate.
int Regex::cand_shortest(const uint8_t* d_text, uint64_t n, uint64_t start, bool* found, uint64_t* end) {
  DeviceDfa* fwd;  // picks the stream, creates the scalars
  if (int rc = ensure(kFwdAnchoredLF, &fwd)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  if (lazy_ && lazy_->done < lazy_->n) {  // host haystack: an anchored run may read to its end
    RB_CUDA(cudaMemcpyAsync(lazy_->dst + lazy_->done, lazy_->src + lazy_->done, lazy_->n - lazy_->done, cudaMemcpyHostToDevice, st));
    lazy_->done = lazy_->n;
  }
  unsigned long long* best = &d_scalars_->cand_best;
  RB_CUDA(cudaMemsetAsync(best, 0xFF, 8, st));
  uint64_t wave = tuning.wave0 ? (tuning.wave0 + 4095) / 4096 * 4096 : 0;
  uint64_t lo = start, b = kNone;
  const uint64_t hi = n + 1;  // candidate positions [start, n]
  stats.scan_redo_rounds = stats.scan_redo_segments = stats.map_passes = stats.waves = 0;
  for (;;) {
    uint64_t limit = hi;
    if (wave && hi - lo > 2 * wave) limit = lo + wave;
    if (int rc = cand_shortest_range(d_text, n, lo, limit, false, best, nullptr)) return rc;
    stats.waves++;
    RB_CUDA(d2h(&b, best, 8));
    if (limit == hi || (b != kNone && b <= limit)) break;
    lo = limit;
    wave *= 16;
  }
  if (b != kNone) { *found = true; *end = b; }
  return 0;
}

int Regex::cand_shortest_range(const uint8_t* d_text, uint64_t n, uint64_t lo, uint64_t hi, bool text_continues, unsigned long long* best,
                               uint32_t* overflow) {
  DeviceDfa* fwd;
  if (int rc = ensure(kFwdAnchoredLF, &fwd)) return rc;
  CandArgs c;
  if (int rc = cand_args(&c)) return rc;
  c.utf8_boundaries = 0;  // the earliest end: an empty match inside a UTF-8 sequence never ends before one at `start`
  const size_t smem = smem_for(fwd->view);
  RB_CUDA(allow_smem(rbgpu::cand_shortest, smem));  // (the kernel, not this member)
  const uint32_t seg = 1024;
  const uint64_t n_seg = (hi - lo + seg - 1) / seg;
  rbgpu::cand_shortest<<<grid_for(n_seg, 256, tuning.blocks_per_sm), 256, smem, (cudaStream_t)stream_>>>(
      fwd->view, smem != 0, c, d_text, n, lo, hi, seg, best, text_continues ? 1 : 0, overflow);
  RB_LAUNCH_CHECK("cand_shortest");
  return 0;
}

// Batched find / find_iter run the unanchored leftmost-first automaton (kind 4), built on first use.  When it is
// over the budget the object switches to candidate starts instead of failing (kind 3 must fit).
int Regex::batch_route(bool* cand) {
  *cand = candidate_mode();
  if (*cand) return 0;
  rb::Error err;
  if (host_dfa(kFwdUnanchoredLF, &err)) return 0;
  if (err.kind != rb::Error::DfaTooBig) return fail(err.msg);
  rb::Error e3;
  if (!host_dfa(kRevAnchoredLongest, &e3)) return fail(err.msg);
  unanchored_too_big_ = true;
  *cand = true;
  return 0;
}

int Regex::cand_batch(int mode, const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint32_t* d_bits, uint64_t* d_spans,
                      uint64_t* d_match_offsets, uint64_t cap) {
  DeviceDfa *fwd, *rev = nullptr;
  if (int rc = ensure(kFwdAnchoredLF, &fwd)) return rc;
  if (mode != 0 && has_looks) if (int rc = ensure(kRevAnchoredLongest, &rev)) return rc;
  CandArgs c;
  if (int rc = cand_args(&c)) return rc;
  BatchArgs a{};
  size_t smem;
  uint32_t per_sm;
  batch_args(&a, d_text, d_offsets, n_rec, fwd, rev, 0, 0, &smem, &per_sm);
  a.out_bits = d_bits;
  a.out_spans = d_spans;
  a.match_offsets = d_match_offsets;
  a.cap = cap;
  cudaStream_t st = (cudaStream_t)stream_;
  static void (*const kBatchCand[4])(BatchArgs, CandArgs) = {batch_cand<0>, batch_cand<1>, batch_cand<2>, batch_cand<3>};
  const auto kernel = kBatchCand[mode];
  RB_CUDA(allow_smem(kernel, smem));
  kernel<<<grid_for(n_rec, 256, tuning.blocks_per_sm), 256, smem, st>>>(a, c);
  RB_LAUNCH_CHECK("batch_cand");
  if (mode <= 1) RB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------ long matches ----
// End of the leftmost-first match anchored at s when it is too long for one thread: the
// anchored automaton over [s, n) in 4 KiB segments, every segment entered in its exact state
// (state maps from EVERY state of the automaton, composed -- the states of `(?s)foo.*bar`
// after `foo` never converge, so no warm-up guess would do), then a maximum over the last match
// positions.  (states + 2) generic passes over the run instead of ~10 s per GiB for one thread.
int Regex::resolve_long_run(const uint8_t* d_text, uint64_t n, uint64_t s, bool text_continues, uint64_t* e_out) {
  DeviceDfa* fwd;
  if (int rc = ensure(kFwdAnchoredLF, &fwd)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  const uint32_t seg = 4096;
  ScanArgs g{};
  g.dfa = fwd->view;
  const size_t smem = smem_for(fwd->view);
  g.use_smem = smem != 0;
  g.text = d_text;
  g.n = n;
  g.base = s;
  g.seg = seg;
  // the start state at s: the look-behind flags come from the bytes next to s (pick_start_fwd)
  uint16_t start_state = fwd->view.start[32];
  if (!fwd->view.uniform_start) {
    uint8_t around[2] = {0, 0};
    const uint64_t lo = s ? s - 1 : 0, hi = std::min(n, s + 1);
    RB_CUDA(d2h(around, d_text + lo, hi - lo));
    const bool has_prev = s > 0, has_cur = s < n;
    const uint8_t prev = has_prev ? around[0] : 0, cur = has_cur ? around[has_prev ? 1 : 0] : 0;
    auto word = [](uint8_t b) { return (b >= 'a' && b <= 'z') || (b >= 'A' && b <= 'Z') || (b >= '0' && b <= '9') || b == '_'; };
    int f = 0;
    if (s == 0) f |= 1;
    if (n == 0) f |= 2 | 8;
    if (s == 0 || prev == '\n') f |= 4;
    const bool last = has_prev && word(prev), cw = has_cur && word(cur);
    f |= (last == cw) ? 32 : 16;
    if (last) f |= 64;
    start_state = fwd->view.start[f];
  }
  // K: the states the run is in at segment boundaries, found as in solve_entries from the run's start state
  // (`(?s)foo.*bar`: 6 of 25 states); it only grows from one window to the next
  uint8_t* present = (uint8_t*)present_.ensure(65536);
  uint16_t* d_first = &d_scalars_->long_entry;
  if (!present) return fail("out of device memory (long run)");
  RB_CUDA(cudaMemsetAsync(present, 0, 65536, st));
  {
    const uint8_t one = 1;
    RB_CUDA(cudaMemcpyAsync(present + start_state, &one, 1, cudaMemcpyHostToDevice, st));
    RB_CUDA(cudaMemcpyAsync(d_first, &start_state, 2, cudaMemcpyHostToDevice, st));
    RB_CUDA(cudaStreamSynchronize(st));
  }
  RB_CUDA(allow_smem(scan_last_match, smem));
  // growing windows from s: a long match is rarely the whole rest of the haystack
  for (uint64_t window = 8ull << 20;; window *= 8) {
    const uint64_t end = window >= n - s ? n : s + window;
    g.limit = end;
    g.n_seg = std::max<uint64_t>(1, (end - s + seg - 1) / seg);
    if (int rc = compose_entries(g, false, d_first)) return rc;
    const uint16_t* exact = (const uint16_t*)exact_.ptr;
    unsigned long long* best = &d_scalars_->long_best;
    RB_CUDA(cudaMemsetAsync(best, 0, 12, st));  // long_best, then long_alive
    scan_last_match<<<grid_for(g.n_seg, 256, tuning.blocks_per_sm), 256, smem, st>>>(g, exact, best, &d_scalars_->long_alive);
    RB_LAUNCH_CHECK("scan_last_match");
    uint32_t h[4] = {0, 0, 0, 0};
    RB_CUDA(d2h(h, best, 12));
    const bool alive = h[2] != 0;
    if (alive && end < n) continue;
    const uint64_t found = (uint64_t)h[0] | ((uint64_t)h[1] << 32);
    if (alive && text_continues) {
      // the run meets the end of a shard's halo: the same verdict as the walk kernels give (err_flag), read
      // by the caller once the search is through
      const uint32_t one = 1;
      RB_CUDA(cudaMemcpyAsync(&d_scalars_->err_flag, &one, 4, cudaMemcpyHostToDevice, st));
      RB_CUDA(cudaStreamSynchronize(st));
      *e_out = found ? found - 1 : n;
      return 0;
    }
    if (found == 0) return fail("internal error: a candidate start has no match (long run)");
    *e_out = found - 1;
    return 0;
  }
}

// ------------------------------------------------- bounded fix-up of entry states --
int Regex::settle_segments(const ScanArgs& a, bool reverse, const std::function<int(uint32_t)>& redo) {
  cudaStream_t st = (cudaStream_t)stream_;
  uint32_t* d_redo = &d_scalars_->list[0];
  for (uint32_t round = 0;; round++) {
    RB_CUDA(cudaMemsetAsync(d_redo, 0, 4, st));
    verify_segments<<<grid_for(a.n_seg, 256, 8), 256, 0, st>>>(a.guess, a.fin, a.n_seg, reverse ? 1 : 0, (uint32_t*)redo_.ptr, d_redo);
    RB_LAUNCH_CHECK("verify_segments");
    RB_CUDA(cudaMemcpyAsync(&h_scalars_->n_redo, d_redo, 4, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    const uint32_t n_redo = h_scalars_->n_redo;
    if (n_redo == 0) return 0;
    if (round == tuning.max_redo_rounds) {
      // wrong guesses keep cascading: solve every entry state at once, then one more redo round
      if (int rc = solve_entries(a, reverse)) return rc;
      continue;
    }
    stats.scan_redo_rounds++;
    stats.scan_redo_segments += n_redo;
    if (int rc = redo(n_redo)) return rc;
  }
}

// Exact entry state of every segment by state-map composition (kernels.cu, "exact entry states"):
// K = the states seen at segment boundaries (guesses and exits); on return fin[] holds, next to
// every segment, the exact state it is entered with, so that one verify + redo round completes
// the scan.  Used when the plain redo rounds do not converge.
int Regex::solve_entries(const ScanArgs& g, bool reverse) {
  cudaStream_t st = (cudaStream_t)stream_;
  const uint64_t n_seg = g.n_seg;
  uint8_t* present = (uint8_t*)present_.ensure(65536);
  if (!present) return fail("out of device memory (state maps)");
  RB_CUDA(cudaMemsetAsync(present, 0, 65536, st));
  mark_states<<<grid_for(n_seg, 256, 8), 256, 0, st>>>(g.guess, n_seg, present);
  RB_LAUNCH_CHECK("mark_states");
  mark_states<<<grid_for(n_seg, 256, 8), 256, 0, st>>>(g.fin, n_seg, present);
  RB_LAUNCH_CHECK("mark_states");
  if (int rc = compose_entries(g, reverse, reverse ? g.guess + (n_seg - 1) : g.guess)) return rc;
  publish_exact<<<grid_for(n_seg, 256, 8), 256, 0, st>>>((const uint16_t*)exact_.ptr, n_seg, reverse ? 1 : 0, g.fin);
  RB_LAUNCH_CHECK("publish_exact");
  return 0;
}

// Run every segment from every state of K (scan_map), add the states the maps lead to, repeat until K is closed;
// then compose the maps along the scan direction: per block of kMapBlock segments, over the blocks from the first
// entry state, and back into every segment.  (|K| + 2) passes over the segments.
int Regex::compose_entries(const ScanArgs& scan_args, bool reverse, const uint16_t* d_entry) {
  ScanArgs g = scan_args;
  cudaStream_t st = (cudaStream_t)stream_;
  const size_t smem = smem_for(g.dfa);
  g.use_smem = smem != 0;
  g.redo_list = nullptr;
  RB_CUDA(allow_smem(scan_map, smem));
  const uint64_t n_seg = g.n_seg;
  const int dir = reverse ? 1 : 0;
  uint8_t* present = (uint8_t*)present_.ptr;
  uint16_t* d_kidx = (uint16_t*)kidx_.ensure(65536 * 2);
  uint32_t* d_new = &d_scalars_->n_new;
  if (!d_kidx) return fail("out of device memory (state maps)");
  std::vector<uint8_t> h_present(65536);
  std::vector<uint16_t> K, kidx;
  uint16_t *d_states = nullptr, *maps = nullptr;
  for (;;) {
    RB_CUDA(d2h(h_present.data(), present, 65536));
    K.clear();
    kidx.assign(65536, 0xFFFF);
    for (uint32_t v = 0; v < g.dfa.n_states; v++)
      if (h_present[v]) { kidx[v] = (uint16_t)K.size(); K.push_back((uint16_t)v); }
    const uint32_t k = (uint32_t)K.size();
    if (k > 512) return fail("the automaton reaches more than 512 distinct states at segment boundaries; state-map composition refused");
    d_states = (uint16_t*)kstates_.ensure(k * 2);
    maps = (uint16_t*)maps_.ensure(n_seg * k * 2);
    if (!d_states || !maps) return fail("out of device memory (state maps)");
    RB_CUDA(cudaMemcpyAsync(d_states, K.data(), k * 2, cudaMemcpyHostToDevice, st));
    RB_CUDA(cudaMemcpyAsync(d_kidx, kidx.data(), 65536 * 2, cudaMemcpyHostToDevice, st));
    scan_map<<<grid_for(n_seg * k, 256, tuning.blocks_per_sm), 256, smem, st>>>(g, dir, d_states, k, maps);
    RB_LAUNCH_CHECK("scan_map");
    stats.map_passes += k;
    RB_CUDA(cudaMemsetAsync(d_new, 0, 4, st));
    closure_check<<<grid_for(n_seg * k, 256, 8), 256, 0, st>>>(maps, n_seg * k, d_kidx, present, d_new);
    RB_LAUNCH_CHECK("closure_check");
    uint32_t n_new = 0;
    RB_CUDA(d2h(&n_new, d_new, 4));  // also orders the host vectors above before they are rebuilt
    if (n_new == 0) break;
  }
  const uint32_t k = (uint32_t)K.size();
  const uint64_t n_blocks = (n_seg + kMapBlock - 1) / kMapBlock;
  uint16_t* comp = (uint16_t*)comp_.ensure(n_blocks * k * 2);
  uint16_t* bentry = (uint16_t*)bentry_.ensure(n_blocks * 2);
  uint16_t* exact = (uint16_t*)exact_.ensure(n_seg * 2);
  if (!comp || !bentry || !exact) return fail("out of device memory (state maps)");
  compose_blocks<<<(uint32_t)((n_blocks * k + 255) / 256), 256, 0, st>>>(maps, d_kidx, d_states, k, n_seg, dir, comp);
  RB_LAUNCH_CHECK("compose_blocks");
  compose_top<<<1, 32, 0, st>>>(comp, d_kidx, k, n_blocks, dir, d_entry, bentry);
  RB_LAUNCH_CHECK("compose_top");
  compose_fill<<<(uint32_t)((n_blocks + 255) / 256), 256, 0, st>>>(maps, d_kidx, k, n_seg, dir, bentry, exact);
  RB_LAUNCH_CHECK("compose_fill");
  return 0;
}

// ------------------------------------------------------------- start bitmap --
Regex::ScanPlan Regex::plan_scan(const uint8_t* d_text, uint64_t base, uint64_t limit, bool fast_table) {
  ScanPlan p;
  const bool utf8_mask = only_utf8 && can_match_empty;
  p.fast = fast_table && !utf8_mask && ((uintptr_t)d_text & 15) == 0 && !tuning.force_generic;
  // segment length: long enough to amortise the warm-up, short enough to fill the GPU
  uint32_t seg = tuning.seg;
  if (seg == 0) {
    const uint64_t lanes = (uint64_t)std::max(1, device_sm_count()) * 1024 * 2;
    uint64_t want = ((limit - base) / lanes + 255) / 256 * 256;
    seg = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(want, 256), p.fast ? 4096 : 1024);
  }
  p.seg = seg;
  p.n_seg = std::max<uint64_t>(1, (limit - base + seg - 1) / seg);
  p.warm = pick_warm(*this);
  if (p.fast) p.warm = (p.warm + 63) / 64 * 64;
  return p;
}

int Regex::scan_starts(const uint8_t* d_text, uint64_t n, uint64_t base, uint64_t limit, ShardIO* io, const ScanPlan& plan,
                       const void* fused_walk) {
  DeviceDfa* rev;
  if (int rc = ensure(kRevUnanchoredAll, &rev)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  const bool utf8_mask = only_utf8 && can_match_empty;
  const bool fast = plan.fast;
  const uint32_t seg = plan.seg;
  const uint64_t n_seg = plan.n_seg;
  if (n_seg >= 0xFFFFFFFFull) return fail("haystack too large for one scan (segment index overflow)");
  ScanArgs a{};
  a.dfa = rev->view;
  a.text = d_text;
  a.n = n;
  a.limit = limit;
  a.base = base;
  a.n_seg = n_seg;
  a.seg = seg;
  a.warm = plan.warm;
  a.bitmap = (uint64_t*)bitmap_.ensure(((n >> 6) + 2) * 8);
  a.guess = (uint16_t*)guess_.ensure(n_seg * 2);
  a.fin = (uint16_t*)fin_.ensure((n_seg + 1) * 2);
  uint32_t* redo = (uint32_t*)redo_.ensure(n_seg * 4);
  if (!a.bitmap || !a.guess || !a.fin || !redo) return fail("out of device memory (scan scratch)");
  a.flag0 = &d_scalars_->flag0;
  a.utf8_boundaries = utf8_mask;
  a.hot = rev->hot;
  size_t smem;
  uint32_t block;
  const WalkArgs* fw = (const WalkArgs*)fused_walk;
  WalkArgs no_walk{};
  // scan_rev_fast<FUSED>: 0 no walk, 1 the fused walk with the table runner, 2 with the fixed-length runner
  static void (*const kScanRevFast[3])(ScanArgs, WalkArgs, CUtensorMap) = {scan_rev_fast<0>, scan_rev_fast<1>, scan_rev_fast<2>};
  const auto rev_fast = kScanRevFast[!fw ? 0 : fw->fixed_len ? 2 : 1];
  if (fast) {
    block = 1024;
    const bool fw_fixed = fw && fw->fixed_len != 0;
    smem = fast_scan_smem(hot_bytes_signed(rev->hot) + (fw && !fw_fixed ? hot_bytes(fw->fwd_hot.n) : 0));
    {  // kernels.cu: rings and mbarriers of the block's warps first, then the tables (hot_signed_below / hot_signed_bytes)
      const uint32_t after_rings = (block / 32) * (2 * 2048 + 64);
      a.tbase_off = after_rings + (uint32_t)hot_bytes(rev->hot.n - rev->hot.match_lo);
      a.fbase_off = after_rings + (uint32_t)hot_bytes_signed(rev->hot);
    }
    RB_CUDA(allow_smem(rev_fast, smem));
  } else {
    smem = smem_for(rev->view);
    a.use_smem = smem != 0;
    block = tuning.block;
    RB_CUDA(allow_smem(scan_rev_bitmap, smem));
  }
  CUtensorMap tmap{};
  if (fast && tuning.tensor_tma && seg >= 64 && seg % 16 == 0 && a.warm <= seg) {
    const uint64_t rows = (n - base) / seg;  // only rows that lie entirely inside the buffer
    if (rows >= 34 && encode_segments(&tmap, d_text + base, seg, rows)) a.tmap_rows = rows;
  }
  auto launch = [&](const ScanArgs& args, uint64_t work) {
    if (fast) rev_fast<<<grid_for(work, block, 1), block, smem, st>>>(args, fw ? *fw : no_walk, tmap);
    else scan_rev_bitmap<<<grid_for(work, block, tuning.blocks_per_sm), block, smem, st>>>(args);
  };
  const bool reuse = io && io->reuse_scan;
  if (!reuse) {
    launch(a, n_seg);
    RB_LAUNCH_CHECK("scan_rev");
  }
  stats.scan_redo_rounds = stats.scan_redo_segments = stats.map_passes = 0;
  ScanArgs r = a;  // a redo round: only the listed segments, each entered with its neighbour's exit
  r.redo_list = redo;
  r.n_redo = &d_scalars_->list[0];
  auto redo_launch = [&](uint32_t n_redo) -> int {
    launch(r, n_redo);
    RB_LAUNCH_CHECK("scan_rev(redo)");
    return 0;
  };
  // A shard may be told the exact state at its top edge by its right neighbour.  A range that starts inside the
  // buffer reports its edge states too: a stream's last piece is checked against the piece before it.
  HostScalars* h = h_scalars_;
  const bool shard = io && (!io->is_first || !io->is_last || io->rev_entry != kNoState || io->own_hi < n || io->own_lo > 0);
  if (shard) {
    RB_CUDA(cudaMemcpyAsync(&h->rev_guess, a.guess + (n_seg - 1), 2, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    io->rev_guess = h->rev_guess;
    if (io->rev_entry != kNoState && io->rev_entry != io->rev_guess) {
      h->seed_state = (uint16_t)io->rev_entry;
      h->seed_seg = (uint32_t)(n_seg - 1);
      h->seed_count = 1;
      RB_CUDA(cudaMemcpyAsync(a.fin + n_seg, &h->seed_state, 2, cudaMemcpyHostToDevice, st));
      RB_CUDA(cudaMemcpyAsync(redo, &h->seed_seg, 4, cudaMemcpyHostToDevice, st));
      RB_CUDA(cudaMemcpyAsync(&d_scalars_->list[0], &h->seed_count, 4, cudaMemcpyHostToDevice, st));
      stats.scan_redo_rounds++;
      stats.scan_redo_segments++;
      if (int rc = redo_launch(1)) return rc;
      io->rev_guess = io->rev_entry;
    }
  }
  if (int rc = settle_segments(a, true, redo_launch)) return rc;
  if (shard) {
    RB_CUDA(cudaMemcpyAsync(&h->rev_left, a.fin, 2, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    io->rev_left = h->rev_left;
  }
  return 0;
}

// ------------------------------------------------------------------ find_all --
// First bitmap bit of a search from `start` (bit i <-> position i + 1), rounded down to the 256-bit shard grain.
static uint64_t shard_own_lo(uint64_t start) { return start ? (start - 1) & ~255ull : 0; }

int Regex::find_all_device(const uint8_t* d_text, uint64_t n, uint64_t start, uint64_t* d_out, uint64_t cap, uint64_t* total) {
  *total = 0;
  if (start > n) return 0;  // re_trait.rs:198-200
  ShardIO io;
  io.own_lo = shard_own_lo(start);
  io.own_hi = n;
  io.chain_p = start;
  io.chain_lm = kNone;
  int rc = find_all_shard_device(d_text, n, &io, d_out, cap);
  *total = io.n_matches;
  return rc;
}

// The paths of a find_iter range, as stats.path reports them, and the chain walk's runners: the kernel tables below are
// indexed by runner.
enum WalkPath { kPathGeneric = 0, kPathFast = 1, kPathFused = 2, kPathPrefilter = 3, kPathCandidates = 4 };
enum WalkRunner { kRunGeneric = 0, kRunTable = 1, kRunFixed = 2 };
using WalkKernel = void (*)(WalkArgs);
using PfKernel = void (*)(WalkArgs, PfArgs, int);

struct Regex::WalkPlan {
  ScanPlan scan;  // the reverse scan of the start bitmap (paths 0-2)
  int path = kPathGeneric;
  // byte-indexed table: uniform start state, 16-byte aligned text; fixed length: no haystack access, so every candidate
  // must be a match start (not with candidate starts), and not as the prefilter's verifier
  int runner = kRunGeneric;
  bool fused = false;  // every lane of the fast scan kernel also walks its own segment (chunk == segment)
  uint32_t chunk = 0;  // bitmap bits per chunk
  size_t smem = 0;     // dynamic shared memory of the runner
  PfArgs pf{};
  WalkKernel walk = nullptr, compact = nullptr, sequential = nullptr;
  PfKernel pf_scan = nullptr;  // the prefilter path, which launches it in place of the three above
};

Regex::WalkPlan Regex::plan_walk(const uint8_t* d_text, const ShardIO& io, const DeviceDfa* fwd, const DeviceDfa* revall) {
  static const WalkKernel kWalkChunks[3] = {walk_chunks<0>, walk_chunks<1>, walk_chunks<2>};
  static const WalkKernel kCompactSpans[3] = {compact_spans<0>, compact_spans<1>, compact_spans<2>};
  static const WalkKernel kWalkSequential[3] = {walk_sequential<0>, walk_sequential<1>, walk_sequential<2>};
  static const PfKernel kLiteralScan[2][4] = {{literal_scan<0, 1>, literal_scan<0, 2>, literal_scan<0, 3>, literal_scan<0, 4>},
                                              {literal_scan<1, 1>, literal_scan<1, 2>, literal_scan<1, 3>, literal_scan<1, 4>}};  // [runner][bytes - 1]
  WalkPlan p;
  const bool cand = candidate_mode();
  const bool aligned = ((uintptr_t)d_text & 15) == 0;
  p.scan = plan_scan(d_text, io.own_lo, io.own_hi,
                     !cand && hot_signed_ok(revall->hot) && fast_scan_smem(hot_bytes_signed(revall->hot)) <= kMaxDynamicSmem);
  const bool table = fwd->hot.n != 0 && fwd->view.uniform_start && aligned && !tuning.force_generic;
  // literal prefilter: no start bitmap at all -- literal_scan finds, verifies and chains the candidates
  const bool pf = tuning.prefilter && !tuning.force_generic && aligned && plan_prefilter() &&
                  (tuning.prefilter >= 2 || pf_freq_ <= kPrefilterAutoFreq);
  const bool fixed = !pf && min_len == max_len && min_len > 0 && !has_looks && !tuning.force_generic && !cand;
  p.runner = fixed ? kRunFixed : table ? kRunTable : kRunGeneric;
  p.fused = !pf && !cand && p.scan.fast && p.runner != kRunGeneric && tuning.fuse && !io.reuse_scan &&
            fast_scan_smem(hot_bytes_signed(revall->hot) + (p.runner == kRunTable ? hot_bytes(fwd->hot.n) : 0)) <= kMaxDynamicSmem;
  p.path = pf ? kPathPrefilter : cand ? kPathCandidates : p.fused ? kPathFused : p.scan.fast ? kPathFast : kPathGeneric;
  p.chunk = pf ? 8192 : p.fused ? p.scan.seg : std::max<uint32_t>(256, (tuning.chunk + 255) / 256 * 256);
  p.smem = p.runner == kRunTable ? hot_bytes(fwd->hot.n) + 256 : p.runner == kRunGeneric ? smem_for(fwd->view) : 0;
  p.walk = kWalkChunks[p.runner];
  p.compact = kCompactSpans[p.runner];
  p.sequential = kWalkSequential[p.runner];
  if (pf) {
    std::memcpy(&p.pf, pf_words_.data(), sizeof p.pf);
    p.pf_scan = kLiteralScan[p.runner][p.pf.n_bytes - 1];
  }
  stats.path = p.path;
  stats.fused = p.fused;
  return p;
}

// ---- stitch: bring the speculative chunk walks into agreement with the sequential iterator (DESIGN.md §2) ----
int Regex::stitch_chunks(WalkArgs* w, const std::function<int(const WalkArgs&, uint32_t)>& rewalk,
                         const std::function<int(const WalkArgs&)>& sequential, ChainKey** grand_key) {
  cudaStream_t st = (cudaStream_t)stream_;
  const uint64_t nc = w->n_chunks, n_blocks = (nc + 1023) / 1024;
  uint32_t* list = d_scalars_->list;
  HostScalars* h = h_scalars_;
  *grand_key = nullptr;
  stats.stitch_rounds = stats.stitch_dirty_chunks = stats.sequential_passes = stats.long_runs = 0;
  if (!has_looks && !can_match_empty) {
    RB_CUDA(cudaMemsetAsync(list, 0, 16, st));
    stitch_fast<<<grid_for(nc, 256, 8), 256, 0, st>>>(*w, list);
    RB_LAUNCH_CHECK("stitch_fast");
    RB_CUDA(cudaMemcpyAsync(h->list, list, 16, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    if (h->list[2] == 0) return 0;  // (a deferred chunk -- long run -- asks for the general loop too)
  }
  ChainKey* excl = (ChainKey*)excl_.ensure(nc * sizeof(ChainKey));
  ChainKey* btot = (ChainKey*)btot_.ensure((n_blocks + 1) * sizeof(ChainKey));
  if (!excl || !btot) return fail("out of device memory (stitch scratch)");
  *grand_key = btot + n_blocks;
  // *w over the dirty list, taken at each use so that it carries the long runs resolved so far
  auto dirty = [&] { WalkArgs d = *w; d.dirty_list = (uint32_t*)dirty_.ptr; d.n_dirty = list; return d; };
  for (uint32_t dirty_rounds = 0;;) {
    RB_CUDA(cudaMemsetAsync(&d_scalars_->first_deferred, 0xFF, 4, st));
    entries_local<<<(uint32_t)n_blocks, 1024, 0, st>>>(*w, excl, btot, &d_scalars_->first_deferred);
    RB_LAUNCH_CHECK("entries_local");
    entries_blocks<<<1, 1024, 0, st>>>(btot, n_blocks, *grand_key);
    RB_LAUNCH_CHECK("entries_blocks");
    RB_CUDA(cudaMemsetAsync(list, 0, 12, st));       // [0] chunks to walk again, [1] changed decisions
    RB_CUDA(cudaMemsetAsync(list + 3, 0xFF, 4, st));  // [3] smallest chunk index to walk again
    stitch_resolve<<<grid_for(nc, 256, 8), 256, 0, st>>>(dirty(), excl, btot, list);
    RB_LAUNCH_CHECK("stitch_resolve");
    RB_CUDA(cudaMemcpyAsync(h->list, list, sizeof h->list + sizeof h->long_req, cudaMemcpyDeviceToHost, st));  // list, long_req
    RB_CUDA(cudaStreamSynchronize(st));
    const uint32_t n_dirty = h->list[0], n_changed = h->list[1];
    const uint64_t long_s = h->long_req;
    bool serve = long_s != kNone;
    if (serve) {
      // the request of a chunk that this round found covered by an earlier match is dropped
      uint32_t m = 0;
      RB_CUDA(d2h(&m, w->meta + (long_s - w->base) / w->chunk, 4));
      serve = (m >> 30) == kChunkDeferred;
      if (!serve) RB_CUDA(cudaMemsetAsync(w->long_req, 0xFF, 8, st));
    }
    if (serve) {
      // a chunk walked from its exact entry met a match longer than kExactRunCap: measure it in parallel,
      // remember it, and let the stitch walk the deferred chunk again
      if (w->n_long == kMaxLongRuns) return fail("more than 256 matches longer than 256 KiB in one search");
      uint64_t e = kNone;
      if (int rc = resolve_long_run(w->text, w->n, long_s, w->text_continues != 0, &e)) return rc;
      const uint64_t pair[2] = {long_s, e};
      RB_CUDA(cudaMemcpyAsync((uint64_t*)long_tab_.ptr + 2 * w->n_long, pair, 16, cudaMemcpyHostToDevice, st));
      RB_CUDA(cudaMemsetAsync(w->long_req, 0xFF, 8, st));
      RB_CUDA(cudaStreamSynchronize(st));
      w->n_long++;
      stats.long_runs++;
    }
    if (n_dirty == 0 && n_changed == 0 && !serve) return 0;
    stats.stitch_rounds++;
    stats.stitch_dirty_chunks += n_dirty;
    if (n_dirty == 0) continue;
    if (++dirty_rounds > tuning.max_stitch_rounds) {
      // chains that do not meet again: one sequential pass from the leftmost such chunk
      WalkArgs s = dirty();
      s.seq_from = h->list[3];
      if (int rc = sequential(s)) return rc;
      stats.sequential_passes++;
      dirty_rounds = 0;
    } else if (int rc = rewalk(dirty(), n_dirty)) {
      return rc;
    }
  }
}

int Regex::find_all_shard_device(const uint8_t* d_text, uint64_t n, ShardIO* io, uint64_t* d_out, uint64_t cap) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  io->n_matches = 0;
  io->halo_overflow = false;
  io->left_ctx_short = false;
  if (is_set_) return fail("find requires exactly one pattern (RegexSet cannot be used with find, exec.rs:510-512)");
  if (io->own_hi > n || io->own_lo > io->own_hi || (io->own_lo & 255) || (!io->is_last && ((io->own_hi & 255) || io->own_hi == n)))
    return fail("bad shard geometry: own_lo/own_hi must be multiples of 256 inside the buffer (own_hi == n only for the last shard)");
  DeviceDfa *fwd, *rev = nullptr, *revall = nullptr;
  if (int rc = ensure(kFwdAnchoredLF, &fwd)) return rc;
  if (has_looks) if (int rc = ensure(kRevAnchoredLongest, &rev)) return rc;
  // candidate-start mode: the start bitmap is a superset of the match starts (cand_bitmap), not the reverse scan's
  if (!candidate_mode()) if (int rc = ensure(kRevUnanchoredAll, &revall)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  cudaEvent_t ev[3] = {(cudaEvent_t)timing_events_[0], (cudaEvent_t)timing_events_[1], (cudaEvent_t)timing_events_[2]};
  RB_CUDA(cudaEventRecord(ev[0], st));
  const WalkPlan plan = plan_walk(d_text, *io, fwd, revall);
  const bool pf = plan.path == kPathPrefilter;
  // literal_scan also has ~9 KB of static shared memory: opt in whenever the sum could pass 48 KB
  if (pf) RB_CUDA(allow_smem(plan.pf_scan, plan.smem, 48 * 1024));
  else for (WalkKernel k : {plan.walk, plan.compact, plan.sequential}) RB_CUDA(allow_smem(k, plan.smem));
  WalkArgs w{};
  w.fwd = fwd->view;
  if (rev) w.rev = rev->view;
  w.text = d_text;
  w.n = n;
  if (!bitmap_.ensure(((n >> 6) + 2) * 8)) return fail("out of device memory (bitmap)");
  w.bitmap = (const uint64_t*)bitmap_.ptr;
  DeviceScalars* ds = d_scalars_;
  w.flag0 = &ds->flag0;
  w.base = io->own_lo;
  w.limit = io->own_hi;
  w.text_continues = !io->is_last;
  w.chunk = plan.chunk;
  w.stage_cap = std::max<uint32_t>(4, w.chunk / 64);
  w.n_chunks = std::max<uint64_t>(1, (w.limit - w.base + w.chunk - 1) / w.chunk);
  const uint64_t nc = w.n_chunks;
  w.in_p = (uint64_t*)in_p_.ensure(nc * 8);
  w.in_lm = (uint64_t*)in_lm_.ensure(nc * 8);
  w.out_p = (uint64_t*)out_p_.ensure(nc * 8);
  w.out_lm = (uint64_t*)out_lm_.ensure(nc * 8);
  w.count = (uint64_t*)count_.ensure(nc * 8);
  uint64_t* offset = (uint64_t*)offset_.ensure(nc * 8);
  const void* dirty_list = dirty_.ensure(nc * 4);  // stitch_chunks
  w.first_cand = (uint64_t*)first_cand_.ensure(nc * 8);
  w.skip = (uint32_t*)skip_.ensure(nc * 4);
  w.meta = (uint32_t*)meta_.ensure(nc * 4);
  w.stage = (uint64_t*)stage_.ensure(nc * (uint64_t)w.stage_cap * 16);
  if (!w.in_p || !w.in_lm || !w.out_p || !w.out_lm || !w.count || !offset || !dirty_list || !w.first_cand || !w.skip || !w.meta || !w.stage)
    return fail("out of device memory (walk scratch)");
  w.offset = offset;
  w.out = d_out;
  w.cap = d_out ? cap : 0;
  w.utf8 = only_utf8;
  w.emulate_slice = has_looks;
  w.can_match_empty = can_match_empty;
  w.use_smem = plan.runner == kRunGeneric && plan.smem != 0;
  if (plan.runner == kRunTable) w.fwd_hot = fwd->hot;
  if (plan.runner == kRunFixed) w.fixed_len = min_len;
  w.err_flag = &ds->err_flag;
  w.floor_flag = &ds->floor_flag;
  // long anchored runs go to resolve_long_run (automata of up to 128 states), requested in long_req
  w.long_tab = (const uint64_t*)long_tab_.ensure(kMaxLongRuns * 16);
  if (!w.long_tab) return fail("out of device memory (long runs)");
  w.exact_cap = fwd->view.n_states <= 128 ? kExactRunCap : kNone;
  w.long_req = &ds->long_req;
  RB_CUDA(cudaMemsetAsync(w.long_req, 0xFF, 8, st));
  w.clamp_p = io->chain_clamped ? io->chain_p : kNone;
  RB_CUDA(cudaMemsetAsync(w.err_flag, 0, 8, st));  // err_flag, floor_flag
  // entry states: chunk 0 starts the real chain at `start`; the rest speculate.
  init_walk_entries<<<grid_for(nc, 256, 8), 256, 0, st>>>(w.in_p, w.in_lm, w.skip, nc, io->chain_p, io->chain_lm);
  RB_LAUNCH_CHECK("init_walk_entries");
  auto launch_pf = [&](const WalkArgs& args, uint64_t chunks, int mode) {  // one warp per chunk
    plan.pf_scan<<<mode == 2 ? 1 : grid_for(chunks * 32, 256, 3), 256, plan.smem, st>>>(args, plan.pf, mode);
  };
  if (plan.path < kPathPrefilter) {
    if (int rc = scan_starts(d_text, n, io->own_lo, io->own_hi, io, plan.scan, plan.fused ? &w : nullptr)) return rc;
  } else {
    if (pf) {
      launch_pf(w, nc, 0);
      RB_LAUNCH_CHECK("literal_scan");
    } else if (int rc = cand_starts(d_text, n, io->own_lo, io->own_hi, !io->is_last)) {
      return rc;
    }
    io->rev_guess = io->rev_entry != kNoState ? io->rev_entry : kPrefilterState;  // no reverse scan, nothing to guess
    io->rev_left = kPrefilterState;
    stats.scan_redo_rounds = stats.scan_redo_segments = stats.map_passes = 0;
  }
  RB_CUDA(cudaEventRecord(ev[1], st));
  if (!pf && !plan.fused) {
    plan.walk<<<grid_for(nc, 256, 6), 256, plan.smem, st>>>(w);
    RB_LAUNCH_CHECK("walk_chunks");
  }
  auto rewalk = [&](const WalkArgs& args, uint32_t n_dirty) {
    if (pf) launch_pf(args, n_dirty, 1);
    else plan.walk<<<grid_for(n_dirty, 256, 6), 256, plan.smem, st>>>(args);
    RB_LAUNCH_CHECK("walk_chunks(dirty)");
    return 0;
  };
  auto sequential = [&](const WalkArgs& args) {
    if (pf) launch_pf(args, 1, 2);
    else plan.sequential<<<1, 256, plan.smem, st>>>(args);
    RB_LAUNCH_CHECK("walk_sequential");
    return 0;
  };
  ChainKey* grand_key;
  if (int rc = stitch_chunks(&w, rewalk, sequential, &grand_key)) return rc;
  unsigned long long* grand;
  if (int rc = prefix_sum(w.count, offset, nc, &grand)) return rc;
  if (w.cap > 0 && pf) {
    compact_staged<<<grid_for(nc, 256, 6), 256, 0, st>>>(w);
    RB_LAUNCH_CHECK("compact_staged");
    launch_pf(w, nc, 3);  // chunks with more matches than staging slots: straight into the output
    RB_LAUNCH_CHECK("literal_scan(overflow)");
  } else if (w.cap > 0) {
    plan.compact<<<grid_for(nc, 256, 6), 256, plan.smem, st>>>(w);
    RB_LAUNCH_CHECK("compact_spans");
  }
  HostScalars* h = h_scalars_;
  RB_CUDA(cudaMemcpyAsync(&h->n_matches, grand, 8, cudaMemcpyDeviceToHost, st));
  if (grand_key) {  // exit state = the last contribution of the whole range
    RB_CUDA(cudaMemcpyAsync(h->exit, grand_key, 16, cudaMemcpyDeviceToHost, st));
  } else {  // the last chunk's exit
    RB_CUDA(cudaMemcpyAsync(&h->exit[0], w.out_p + (nc - 1), 8, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaMemcpyAsync(&h->exit[1], w.out_lm + (nc - 1), 8, cudaMemcpyDeviceToHost, st));
  }
  RB_CUDA(cudaMemcpyAsync(&h->err_flag, w.err_flag, 8, cudaMemcpyDeviceToHost, st));  // err_flag, floor_flag
  RB_CUDA(cudaEventRecord(ev[2], st));
  RB_CUDA(cudaStreamSynchronize(st));
  io->n_matches = h->n_matches;
  // ChainKey: p + 1; 0 = nothing in this range moved the iterator (speculative shard without candidates), ~0 = the end
  const uint64_t* x = h->exit;
  io->exit_p = !grand_key ? x[0] : x[0] == 0 ? kSpec : x[0] == kNone ? kNone : x[0] - 1;
  io->exit_lm = grand_key && x[0] == 0 ? kNone : x[1];
  io->halo_overflow = h->err_flag != 0;
  io->left_ctx_short = h->floor_flag != 0;
  cudaEventElapsedTime(&stats.scan_ms, ev[0], ev[1]);
  cudaEventElapsedTime(&stats.walk_ms, ev[1], ev[2]);
  cudaEventElapsedTime(&stats.total_ms, ev[0], ev[2]);
  if (io->halo_overflow) return fail("a match runs past the end of the shard halo; enlarge the halo");
  if (io->left_ctx_short)
    return fail("the reverse-on-slice scan of a look-around pattern reaches the start of the shard buffer; enlarge the left context");
  return 0;
}

int Regex::find_at_device(const uint8_t* d_text, uint64_t n, uint64_t start, bool* found, uint64_t* s, uint64_t* e) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *found = false;
  uint64_t* d_out = (uint64_t*)out_.ensure(16);
  if (!d_out) return fail("out of device memory");
  uint64_t total = 0;
  // The first element of the find_iter chain started at `start` is find_at(start).
  if (int rc = find_all_device(d_text, n, start, d_out, 1, &total)) return rc;
  if (total == 0) return 0;
  uint64_t h[2];
  RB_CUDA(cudaMemcpyAsync(h, d_out, 16, cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
  RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  *found = true;
  *s = h[0];
  *e = h[1];
  return 0;
}

// ------------------------------------------------------ forward reductions ----
// One wave of a forward all-match scan: positions [start, limit) of the haystack (limit == n + 1
// includes the end-of-text step), entered in state `entry` (kNoEntry: the start state for the
// flags at `start`).  result_host[0] = first match end, [1..] = OR of the pattern masks;
// *exit_state = exact state after the last position (the next wave's entry).
int Regex::forward_range(const uint8_t* d_text, uint64_t n, uint64_t start, uint64_t limit, uint32_t entry, bool want_masks,
                         uint64_t* result_host, uint32_t* exit_state) {
  DeviceDfa* fwd;
  if (int rc = ensure(kFwdUnanchoredAll, &fwd)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  // fast path (scan_fwd_fast): hot table, 16-byte aligned haystack and start; RegexSets only when
  // matches are known to be rare (a narrowed set, see forward_reduce): the fast kernel finds the
  // patterns of a match by redoing that 64-byte group on the full table
  const bool fast_ok = (!want_masks || sparse_set_) && fwd->hot.n != 0 && !tuning.force_generic && tuning.tensor_tma && encode_tiled() &&
                       ((uintptr_t)d_text & 15) == 0 && (start & 63) == 0 &&
                       fast_scan_smem(hot_bytes(fwd->hot.n)) <= kMaxDynamicSmem;
  const uint32_t seg = tuning.seg ? tuning.seg : (fast_ok ? 4096 : 1024);
  const uint64_t n_seg = (limit - start + seg - 1) / seg;
  if (n_seg >= 0xFFFFFFFFull) return fail("haystack too large for one scan (segment index overflow)");
  const uint32_t mw = fwd->view.mask_words;
  ScanArgs a{};
  a.dfa = fwd->view;
  const size_t smem = smem_for(fwd->view);
  a.use_smem = smem != 0;
  a.text = d_text;
  a.n = n;
  a.base = start;
  a.fwd_limit = limit;
  a.entry0 = entry;
  a.n_seg = n_seg;
  a.seg = seg;
  a.warm = pick_warm(*this);
  if (fast_ok) a.warm = (a.warm + 63) / 64 * 64;
  a.seg_first = (uint64_t*)seg_first_.ensure(n_seg * 8);
  a.seg_mask = want_masks ? (uint64_t*)seg_mask_.ensure(n_seg * 8 * mw) : nullptr;
  a.guess = (uint16_t*)guess_.ensure(n_seg * 2);
  a.fin = (uint16_t*)fin_.ensure(n_seg * 2);
  uint32_t* redo = (uint32_t*)redo_.ensure(n_seg * 4);
  if (!a.seg_first || (want_masks && !a.seg_mask) || !a.guess || !a.fin || !redo)
    return fail("out of device memory (scan scratch)");
  RB_CUDA(allow_smem(scan_fwd_reduce, smem));
  // whole warps of full segments go to the fast kernel; segment 0, the ragged end and the EOF step stay generic
  const uint64_t n_full = (std::min(limit, n) - start) / seg;
  bool fast_launched = false;
  if (!fork_event_) {
    cudaEvent_t e1, e2;
    RB_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
    RB_CUDA(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
    fork_event_ = e1;
    join_event_ = e2;
  }
  if (fast_ok && seg % 64 == 0 && a.warm <= seg && n_full >= 34) {
    const uint64_t skip_lo = 1, skip_hi = 1 + (n_full - 1) / 32 * 32;
    CUtensorMap tmap{};
    // row 0 = segment skip_lo - 1 (warm-up source of the first warp)
    if (encode_segments(&tmap, d_text + start + (skip_lo - 1) * (uint64_t)seg, seg, skip_hi - skip_lo + 1)) {
      a.hot = fwd->hot;
      a.skip_lo = skip_lo;
      a.skip_hi = skip_hi;
      const size_t fsm = fast_scan_smem(hot_bytes(fwd->hot.n));
      RB_CUDA(allow_smem(scan_fwd_fast, fsm));
      RB_CUDA(cudaEventRecord((cudaEvent_t)fork_event_, st));  // the side stream starts once everything before this point is done
      scan_fwd_fast<<<grid_for(skip_hi - skip_lo, 1024, 1), 1024, fsm, st>>>(a, tmap);
      RB_LAUNCH_CHECK("scan_fwd_fast");
      fast_launched = true;
    }
  }
  // The generic kernel takes what the fast one leaves (segment 0, the ragged end, the end-of-text
  // step): a handful of 4 KiB segments walked by single threads, ~0.25 ms of pure latency (ncu
  // profiles/r02: 10 % issue, 3 % of the warps).  It runs beside the fast kernel on a second stream.
  if (fast_launched) {
    if (int rc = side_streams()) return rc;
    cudaStream_t side = (cudaStream_t)back_stream_;
    RB_CUDA(cudaStreamWaitEvent(side, (cudaEvent_t)fork_event_, 0));
    scan_fwd_reduce<<<grid_for(n_seg, tuning.block, tuning.blocks_per_sm), tuning.block, smem, side>>>(a);
    RB_LAUNCH_CHECK("scan_fwd_reduce");
    RB_CUDA(cudaEventRecord((cudaEvent_t)join_event_, side));
    RB_CUDA(cudaStreamWaitEvent(st, (cudaEvent_t)join_event_, 0));
  } else {
    scan_fwd_reduce<<<grid_for(n_seg, tuning.block, tuning.blocks_per_sm), tuning.block, smem, st>>>(a);
    RB_LAUNCH_CHECK("scan_fwd_reduce");
  }
  ScanArgs r = a;
  r.redo_list = redo;
  r.n_redo = &d_scalars_->list[0];
  auto redo_launch = [&](uint32_t n_redo) -> int {
    scan_fwd_reduce<<<grid_for(n_redo, tuning.block, tuning.blocks_per_sm), tuning.block, smem, st>>>(r);
    RB_LAUNCH_CHECK("scan_fwd_reduce(redo)");
    return 0;
  };
  if (int rc = settle_segments(a, false, redo_launch)) return rc;
  unsigned long long* result = d_scalars_->fwd_result;
  uint64_t* h = h_scalars_->fwd_result;
  h[0] = kNone;
  for (uint32_t w = 0; w < kMaxMaskWords; w++) h[1 + w] = 0;
  RB_CUDA(cudaMemcpyAsync(result, h, 8 * (1 + kMaxMaskWords), cudaMemcpyHostToDevice, st));
  reduce_segments<<<grid_for(n_seg, 256, 4), 256, 0, st>>>(a.seg_first, a.seg_mask, n_seg, mw, result);
  RB_LAUNCH_CHECK("reduce_segments");
  RB_CUDA(cudaMemcpyAsync(h, result, 8 * (1 + kMaxMaskWords), cudaMemcpyDeviceToHost, st));
  RB_CUDA(cudaMemcpyAsync(&h_scalars_->fwd_exit, a.fin + (n_seg - 1), 2, cudaMemcpyDeviceToHost, st));
  RB_CUDA(cudaStreamSynchronize(st));
  for (uint32_t w = 0; w < 1 + kMaxMaskWords; w++) result_host[w] = h[w];
  *exit_state = h_scalars_->fwd_exit;
  return 0;
}

// is_match / shortest_match / RegexSet::matches over one haystack, in waves of growing size
// (64 MiB, x16 each) so that the search stops early the way the reference does:
//   - a single pattern stops at the first wave that holds a match (dfa.rs:658-667, quit_after_match);
//   - a set stops once every pattern has matched (dfa.rs:675-682);
//   - a set ALSO narrows: patterns that matched in the first waves need no further tracking,
//     so the rest of the haystack is scanned with the automaton of the patterns that are still
//     open (usually a handful of rare ones: small, shared-memory resident, fast kernel) instead
//     of the product automaton of all of them.  That automaton knows nothing about the bytes
//     already passed, so it scans from `start` again; narrowing happens after the first two
//     waves only, which bounds the repeated work to 1/16 of the haystack.
// end: positions [start, end) are searched (n + 1 = to the end of the text, the default); entry:
// exact automaton state at `start` (a shard, kNoEntry = a fresh search); *exit_state: the exact
// state after the last position (what the right-hand shard must be entered with).
int Regex::forward_reduce(const uint8_t* d_text, uint64_t n, uint64_t start, bool want_masks, uint64_t* result_host, uint64_t end,
                          uint32_t entry, uint32_t* exit_out) {
  const uint32_t n_pat = (uint32_t)patterns_.size();
  const uint32_t rw = result_words() - 1;
  result_host[0] = kNone;
  for (uint32_t w = 0; w < rw; w++) result_host[1 + w] = 0;
  if (int rc = init_device()) return rc;
  // The automata of this search: the product automaton, or one per pattern group.  Every wave runs each group that
  // is still open over the same positions; each group carries its own state into the next wave.
  if (!groups_.empty() && (entry != kNoEntry || end != ~0ull)) return fail("a RegexSet searched in pattern groups cannot be searched in shards");
  std::vector<Regex*> tabs;
  std::vector<uint32_t> firsts;
  forward_tabs(&tabs, &firsts);
  const uint32_t n_tab = (uint32_t)tabs.size();
  std::vector<uint32_t> entries(n_tab, entry);
  std::vector<char> done(n_tab, 0);
  uint64_t wave = tuning.wave0 ? (tuning.wave0 + 4095) / 4096 * 4096 : 0;
  uint64_t lo = start;
  end = std::min(end, n + 1);
  const bool whole = end == n + 1 && entry == kNoEntry;  // narrowing restarts the search at `start` with a fresh automaton
  if (exit_out) *exit_out = entry == kNoEntry ? kNoState : entry;
  stats.scan_redo_rounds = stats.scan_redo_segments = stats.map_passes = stats.waves = 0;
  stats.groups = n_tab;
  std::vector<uint64_t> before(rw);
  for (uint32_t wi = 0;; wi++) {
    uint64_t limit = end;
    if (wave && end - lo > 2 * wave) limit = (lo + wave) / 4096 * 4096;
    if (lazy_) {  // host haystack: bring in what this wave reads (plus a little for the flags at its end)
      const uint64_t want = std::min(lazy_->n, limit + 64);
      if (want > lazy_->done) {
        RB_CUDA(cudaMemcpyAsync(lazy_->dst + lazy_->done, lazy_->src + lazy_->done, want - lazy_->done, cudaMemcpyHostToDevice, (cudaStream_t)stream_));
        lazy_->done = want;
      }
    }
    std::copy(result_host + 1, result_host + 1 + rw, before.begin());
    bool live = false;
    if (int rc = forward_step(tabs, firsts, d_text, n, lo, limit, want_masks, &entries, &done, result_host, &live)) return rc;
    if (exit_out) *exit_out = entries[0];  // (shards have one automaton)
    stats.waves++;
    bool fresh = false;
    for (uint32_t w = 0; w < rw; w++) fresh = fresh || (result_host[1 + w] & ~before[w]);
    if (limit == end) break;
    if (!want_masks && result_host[0] != kNone) break;
    if (!live) break;
    if (want_masks) {
      std::vector<uint32_t> open;
      for (uint32_t i = 0; i < n_pat; i++)
        if (!((result_host[1 + i / 64] >> (i % 64)) & 1)) open.push_back(i);
      if (open.empty()) break;
      if (tuning.narrow_sets && whole && wi < 2 && fresh && open.size() < n_pat) {
        Regex* sub = nullptr;
        if (int rc = subset(open, &sub)) return rc;
        std::vector<uint64_t> sr(sub->result_words());
        sub->tuning.wave0 = tuning.wave0;
        sub->set_stream(stream_);
        sub->lazy_ = lazy_;
        std::lock_guard<std::recursive_mutex> lock(sub->mu_);
        const int src = sub->forward_reduce(d_text, n, start, true, sr.data());
        sub->lazy_ = nullptr;
        if (src) return fail(sub->last_error());
        stats.waves += sub->stats.waves;
        for (uint32_t j = 0; j < open.size(); j++)
          if ((sr[1 + j / 64] >> (j % 64)) & 1) result_host[1 + open[j] / 64] |= 1ull << (open[j] % 64);
        break;
      }
      retire_matched(firsts, result_host, &done);
    }
    lo = limit;
    wave *= 16;
  }
  return 0;
}

void Regex::forward_tabs(std::vector<Regex*>* tabs, std::vector<uint32_t>* firsts) {
  tabs->assign(1, this);
  firsts->assign(1, 0);
  if (groups_.empty()) return;
  tabs->clear();
  for (auto& g : groups_) {
    g->tuning = tuning;
    g->sparse_set_ = sparse_set_;
    g->set_stream(stream_);
    tabs->push_back(g.get());
  }
  *firsts = group_first_;
}

int Regex::forward_step(const std::vector<Regex*>& tabs, const std::vector<uint32_t>& firsts, const uint8_t* d_text, uint64_t n, uint64_t lo,
                        uint64_t limit, bool want_masks, std::vector<uint32_t>* entries, std::vector<char>* done, uint64_t* result_host,
                        bool* live) {
  const uint32_t rw = result_words() - 1;
  *live = false;
  for (uint32_t g = 0; g < tabs.size(); g++) {
    if ((*done)[g]) continue;
    uint64_t r[1 + kMaxMaskWords];
    uint32_t exit_state = 0;
    if (int rc = tabs[g]->forward_range(d_text, n, lo, limit, (*entries)[g], want_masks, r, &exit_state))
      return tabs[g] == this ? rc : fail(tabs[g]->last_error());
    result_host[0] = std::min(result_host[0], r[0]);
    // group-local mask bit j is pattern firsts[g] + j
    const uint32_t w0 = firsts[g] / 64, sh = firsts[g] % 64;
    for (uint32_t w = 0; w < kMaxMaskWords && w0 + w < rw; w++) {
      result_host[1 + w0 + w] |= r[1 + w] << sh;
      if (sh && w0 + w + 1 < rw) result_host[2 + w0 + w] |= r[1 + w] >> (64 - sh);
    }
    (*entries)[g] = exit_state;
    if (exit_state == 0) (*done)[g] = 1;  // dead state: an anchored search that can no longer match
    *live = *live || !(*done)[g];
  }
  return 0;
}

// a group whose patterns have all matched needs no further search
void Regex::retire_matched(const std::vector<uint32_t>& firsts, const uint64_t* result_host, std::vector<char>* done) const {
  const uint32_t n_tab = (uint32_t)firsts.size(), n_pat = (uint32_t)patterns_.size();
  for (uint32_t g = 0; g < n_tab && n_tab > 1; g++) {
    const uint32_t hi = g + 1 < n_tab ? firsts[g + 1] : n_pat;
    bool all = true;
    for (uint32_t i = firsts[g]; i < hi && all; i++) all = (result_host[1 + i / 64] >> (i % 64)) & 1;
    if (all) (*done)[g] = 1;
  }
}

// ------------------------------------------------------------ pattern groups --
// One group: the set-mode Regex of patterns [lo, hi) with one product automaton (or the error of its determinization).
Regex* Regex::compile_group(const std::vector<std::string>& all, uint32_t lo, uint32_t hi, const CompileOptions& opt, rb::Error* err) {
  const std::vector<std::string> pats(all.begin() + lo, all.begin() + hi);
  CompileOptions o = opt;
  o.as_set = true;
  const std::vector<uint32_t> one{0};
  return compile_impl(pats, o, err, &one, 0);
}

// Groups for [lo, hi): the range itself when its automaton fits (and it is not known not to), else its two halves.
// Ranges of more than 64 patterns split on a multiple of 64 so that large groups own whole mask words.  A single
// pattern over budget fails with its determinization's error.
bool Regex::plan_range(uint32_t lo, uint32_t hi, bool known_too_big, std::vector<std::unique_ptr<Regex>>* out,
                       std::vector<uint32_t>* firsts, rb::Error* err) {
  if (!known_too_big) {
    rb::Error e;
    if (Regex* g = compile_group(patterns_, lo, hi, opt_, &e)) {
      out->emplace_back(g);
      firsts->push_back(lo);
      return true;
    }
    if (e.kind != rb::Error::DfaTooBig || hi - lo == 1) { *err = e; return false; }
  }
  const uint32_t n = hi - lo;
  uint32_t mid = lo + n / 2;
  if (n > 64) {
    mid = (lo + n / 2 + 32) / 64 * 64;
    if (mid <= lo) mid += 64;
    if (mid >= hi) mid -= 64;
  }
  return plan_range(lo, mid, false, out, firsts, err) && plan_range(mid, hi, false, out, firsts, err);
}

// Replaces the group plan: `plan` = the first pattern of each group, compiled as given; else chunks of `chunk`
// patterns split by the budget (the first chunk is known to be over budget when `first_too_big`).  One resulting
// group is the product automaton.  On failure the object is unchanged.
bool Regex::build_groups(const std::vector<uint32_t>* plan, uint32_t chunk, bool first_too_big, rb::Error* err) {
  const uint32_t n = (uint32_t)patterns_.size();
  std::vector<std::unique_ptr<Regex>> gs;
  std::vector<uint32_t> firsts;
  if (plan) {
    for (size_t i = 0; i < plan->size(); i++) {
      const uint32_t lo = (*plan)[i], hi = i + 1 < plan->size() ? (*plan)[i + 1] : n;
      Regex* g = compile_group(patterns_, lo, hi, opt_, err);
      if (!g) return false;
      gs.emplace_back(g);
      firsts.push_back(lo);
    }
  } else {
    for (uint32_t lo = 0; lo < n; lo += chunk)
      if (!plan_range(lo, std::min(n, lo + chunk), lo == 0 && first_too_big, &gs, &firsts, err)) return false;
  }
  subsets_.clear();
  if (gs.size() == 1) {
    host_[kFwdUnanchoredAll] = std::move(gs[0]->host_[kFwdUnanchoredAll]);
    product_fits_ = true;
    groups_.clear();
    group_first_.clear();
    return true;
  }
  groups_ = std::move(gs);
  group_first_ = std::move(firsts);
  return true;
}

int Regex::set_group_patterns(uint32_t k) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (!is_set_) return fail("set_group_patterns applies to a RegexSet");
  if (patterns_.empty()) return 0;  // an empty set has no automaton and nothing to group
  if (k == 0 && product_fits_) {
    groups_.clear();
    group_first_.clear();
    subsets_.clear();
    return 0;
  }
  rb::Error err;
  const uint32_t cap = 64 * kMaxMaskWords;
  if (!build_groups(nullptr, k ? std::min(k, cap) : cap, k == 0 && patterns_.size() <= cap, &err)) return fail("set_group_patterns: " + err.msg);
  return 0;
}

// The RegexSet of a subset of this set's patterns (cached; used by forward_reduce's narrowing).
int Regex::subset(const std::vector<uint32_t>& members, Regex** out) {
  auto it = subsets_.find(members);
  if (it == subsets_.end()) {
    std::vector<std::string> pats;
    for (uint32_t i : members) pats.push_back(patterns_[i]);
    CompileOptions o = opt_;
    o.as_set = true;
    rb::Error err;
    std::unique_ptr<Regex> sub(Regex::compile(pats, o, &err));
    if (!sub) return fail("narrowed pattern set: " + err.msg);
    sub->sparse_set_ = true;
    sub->tuning = tuning;
    it = subsets_.emplace(members, std::move(sub)).first;
  }
  *out = it->second.get();
  return 0;
}


int Regex::shortest_match_device(const uint8_t* d_text, uint64_t n, uint64_t start, bool* found, uint64_t* end) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *found = false;
  if (patterns_.empty() || start > n) return 0;
  if (candidate_mode()) return cand_shortest(d_text, n, start, found, end);
  std::vector<uint64_t> res(result_words());
  if (int rc = forward_reduce(d_text, n, start, false, res.data())) return rc;
  if (res[0] != kNone) { *found = true; *end = res[0]; }
  return 0;
}

int Regex::set_matches_device(const uint8_t* d_text, uint64_t n, uint64_t start, bool* any, uint64_t* masks) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *any = false;
  const uint32_t mw = (uint32_t)((patterns_.size() + 63) / 64);
  for (uint32_t w = 0; w < mw; w++) masks[w] = 0;
  if (patterns_.empty() || start > n) return 0;
  std::vector<uint64_t> res(result_words());
  if (int rc = forward_reduce(d_text, n, start, true, res.data())) return rc;
  for (uint32_t w = 0; w < mw; w++) { masks[w] = res[1 + w]; if (res[1 + w]) *any = true; }
  return 0;
}

// One byte-range shard of a forward search (is_match / shortest_match / RegexSet::matches over a
// sharded haystack; SURVEY.md 8e).  The automaton state flows left to right: a shard that is not
// told its entry state guesses it by running the automaton over the left context in front of
// own_lo (host side, <= 256 bytes) from the start state that belongs to that position; the
// ranks compare each guess with the left neighbour's exact exit state and search again when
// they differ (regex_b200/sharded.py: forward_sharded).
int Regex::forward_shard_device(const uint8_t* d_text, uint64_t n, uint64_t own_lo, uint64_t own_hi, bool is_first, bool is_last, uint32_t entry,
                                bool want_masks, bool* found, uint64_t* first_end, uint64_t* masks, uint32_t* entry_used,
                                uint32_t* exit_state) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *found = false;
  *first_end = kNone;
  const uint32_t mw = (uint32_t)std::max<size_t>(1, (patterns_.size() + 63) / 64);
  for (uint32_t w = 0; w < mw; w++) masks[w] = 0;
  *entry_used = *exit_state = entry;
  if (patterns_.empty()) return 0;
  if (own_lo > own_hi || own_hi > n) return fail("bad shard geometry");
  if (candidate_mode())
    return fail("sharded shortest_match / is_match is not available for a pattern searched from candidate starts (its unanchored "
                "automaton exceeds the DFA table budget); use shortest_match on the whole haystack");
  if (!groups_.empty())
    return fail("sharded RegexSet searches are not available for a set searched in " + std::to_string(groups_.size()) +
                " pattern groups (the shard protocol carries one automaton state and at most 256 pattern bits); use "
                "set_matches on the whole haystack");
  DeviceDfa* fwd;
  if (int rc = ensure(kFwdUnanchoredAll, &fwd)) return rc;
  if (entry == kNoEntry && own_lo > 0) {
    rb::Error err;
    const rb::Dfa* h = host_dfa(kFwdUnanchoredAll, &err);
    if (!h) return fail(err.msg);
    // run the automaton over the last <= 255 bytes in front of own_lo; its start state takes the
    // flags of a position inside a long text (dfa.rs:1415-1434), so one more byte is looked at
    uint64_t from = own_lo > 255 ? own_lo - 255 : 0;
    if (from == 0 && !is_first) from = 1;            // buffer byte 0 is not the start of the haystack
    const uint64_t copy_lo = from ? from - 1 : 0;
    const uint64_t copy_n = std::min<uint64_t>(n, own_lo + 1) - copy_lo;
    std::vector<uint8_t> left(copy_n + 1, 0);
    RB_CUDA(d2h(left.data(), d_text + copy_lo, copy_n));
    uint32_t st = h->start[rb::start_flag_index_forward(left.data(), copy_n, from - copy_lo) & 127];
    for (uint64_t i = from; i < own_lo; i++) st = h->next((uint16_t)st, left[i - copy_lo]);
    entry = st;
  }
  *entry_used = entry;
  std::vector<uint64_t> res(result_words());
  const uint64_t end = is_last ? n + 1 : own_hi;
  if (int rc = forward_reduce(d_text, n, own_lo, want_masks, res.data(), end, entry, exit_state)) return rc;
  if (res[0] != kNone) { *found = true; *first_end = res[0]; }
  for (uint32_t w = 0; w < mw; w++) { masks[w] = res[1 + w]; if (want_masks && res[1 + w]) *found = true; }
  return 0;
}

// -------------------------------------------------------------------- batch ----
bool Regex::batch_args(BatchArgs* a, const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, DeviceDfa* fwd, DeviceDfa* rev,
                       size_t reserve, uint32_t max_per_sm, size_t* smem, uint32_t* per_sm) {
  a->fwd = fwd->view;
  if (rev) a->rev = rev->view;
  *smem = smem_for(fwd->view);
  a->use_smem = *smem != 0;
  a->text = d_text;
  a->offsets = d_offsets;
  a->n_rec = n_rec;
  a->utf8 = only_utf8 ? 1 : 0;
  *per_sm = 0;
  if (!max_per_sm || !fwd->hot.n || (rev && !rev->hot.n) || ((uintptr_t)d_text & 15) != 0 || tuning.force_generic) return false;
  a->fwd_hot = fwd->hot;
  a->fwd_g = (const DfaView*)fwd->view_dev;
  *smem = hot_bytes(fwd->hot.n) + 256;
  if (rev) {
    a->rev_hot = rev->hot;
    a->rev_g = (const DfaView*)rev->view_dev;
    *smem += hot_bytes(rev->hot.n);
  }
  *per_sm = (uint32_t)std::max<size_t>(1, std::min<size_t>(max_per_sm, (220 * 1024) / (*smem + reserve)));
  return true;
}

int Regex::is_match_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint32_t* d_bits) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (n_rec == 0) return 0;
  if (patterns_.empty()) {
    if (int rc = init_device()) return rc;
    RB_CUDA(cudaMemsetAsync(d_bits, 0, (n_rec + 31) / 32 * 4, (cudaStream_t)stream_));
    RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    return 0;
  }
  if (candidate_mode()) return cand_batch(0, d_text, d_offsets, n_rec, d_bits, nullptr, nullptr, 0);
  DeviceDfa* fwd;
  if (int rc = ensure(kFwdUnanchoredAll, &fwd)) return rc;
  BatchArgs a{};
  size_t smem;
  uint32_t per_sm;
  const bool hot = batch_args(&a, d_text, d_offsets, n_rec, fwd, nullptr, 8192, 4, &smem, &per_sm);
  a.out_bits = d_bits;
  if (hot) {
    // tasks of 96..2048 records, at least four per warp of the grid; smaller batches keep one record per lane
    const uint32_t grid0 = grid_for(n_rec, 512, per_sm);
    const uint64_t per_task = n_rec / ((uint64_t)grid0 * 16 * 4);
    a.task_recs = (uint32_t)std::min<uint64_t>(2048, per_task / 32 * 32);
    if (tuning.batch_refill >= 2) a.task_recs = std::max<uint32_t>(a.task_recs, 32);  // tests: whatever the size
    if (tuning.batch_refill && a.task_recs >= (tuning.batch_refill >= 2 ? 32u : 96u)) {
      a.task_counter = &d_scalars_->task_counter;
      RB_CUDA(cudaMemsetAsync(a.task_counter, 0, 8, (cudaStream_t)stream_));
      // (8 KB of static shared memory for the result words on top of the table: opt in whenever the sum may pass 48 KB)
      RB_CUDA(allow_smem(batch_refill, smem, 48 * 1024));
      batch_refill<<<grid_for(n_rec, 512, per_sm), 512, smem, (cudaStream_t)stream_>>>(a);
      RB_LAUNCH_CHECK("batch_refill");
    } else {
      RB_CUDA(allow_smem(batch_fast<0>, smem));
      batch_fast<0><<<grid_for(n_rec, 512, per_sm), 512, smem, (cudaStream_t)stream_>>>(a);
      RB_LAUNCH_CHECK("batch_fast<0>");
    }
  } else {
    RB_CUDA(allow_smem(is_match_batch, smem));
    is_match_batch<<<(uint32_t)((n_rec + 255) / 256), 256, smem, (cudaStream_t)stream_>>>(a);
    RB_LAUNCH_CHECK("is_match_batch");
  }
  RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  return 0;
}

int Regex::find_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_spans, uint32_t* d_bits) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (n_rec == 0) return 0;
  if (is_set_) return fail("find requires exactly one pattern");
  bool cand;
  if (int rc = batch_route(&cand)) return rc;
  if (cand) return cand_batch(1, d_text, d_offsets, n_rec, d_bits, d_spans, nullptr, 0);
  DeviceDfa *fwd, *rev;
  if (int rc = ensure(kFwdUnanchoredLF, &fwd)) return rc;
  if (int rc = ensure(kRevAnchoredLongest, &rev)) return rc;
  BatchArgs a{};
  size_t smem;
  uint32_t per_sm;
  const bool hot = batch_args(&a, d_text, d_offsets, n_rec, fwd, rev, 16384, 4, &smem, &per_sm);
  a.out_bits = d_bits;
  a.out_spans = d_spans;
  if (hot) {
    RB_CUDA(allow_smem(batch_fast<1>, smem));
    batch_fast<1><<<grid_for(n_rec, 512, per_sm), 512, smem, (cudaStream_t)stream_>>>(a);
    RB_LAUNCH_CHECK("batch_fast<1>");
  } else {
    find_batch<<<(uint32_t)((n_rec + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(a);
    RB_LAUNCH_CHECK("find_batch");
  }
  RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  return 0;
}

// find_iter per record into a CSR list: count pass, in-place exclusive scan of the counts (entry n_rec = the
// total), write pass (kernels.cu batch_iter).
int Regex::find_iter_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_match_offsets,
                                  uint64_t* d_out, uint64_t cap, uint64_t* total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  return iter_batch(d_text, d_offsets, n_rec, d_match_offsets, d_out, cap, total, nullptr);
}

int Regex::iter_batch(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_match_offsets, uint64_t* d_out,
                      uint64_t cap, uint64_t* total, DeviceBuf* grow) {
  *total = 0;
  if (is_set_) return fail("find requires exactly one pattern");
  bool cand;
  if (int rc = batch_route(&cand)) return rc;
  DeviceDfa *fwd, *rev;
  if (int rc = ensure(cand ? kFwdAnchoredLF : kFwdUnanchoredLF, &fwd)) return rc;
  if (int rc = ensure(kRevAnchoredLongest, &rev)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_rec == 0) {
    RB_CUDA(cudaMemsetAsync(d_match_offsets, 0, 8, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  BatchArgs a{};
  size_t fsm;
  uint32_t per_sm;
  // __launch_bounds__(512, 2): two blocks per SM fit the registers of the iterator
  const bool fast = batch_args(&a, d_text, d_offsets, n_rec, fwd, rev, 16384, cand ? 0 : 2, &fsm, &per_sm);
  a.match_offsets = d_match_offsets;
  a.out_spans = d_out;
  a.cap = d_out ? cap : 0;
  uint32_t grid = (uint32_t)((n_rec + 255) / 256);
  if (fast) {
    grid = grid_for(n_rec, 512, per_sm);
    RB_CUDA(allow_smem(batch_iter_fast<0>, fsm));
    RB_CUDA(allow_smem(batch_iter_fast<1>, fsm));
  }
  // ---- count ----
  a.fwd_only = !can_match_empty && !has_looks && !cand;  // (the forward-only count needs kind 4)
  RB_CUDA(cudaMemsetAsync(d_match_offsets + n_rec, 0, 8, st));
  if (cand) {
    if (int rc = cand_batch(2, d_text, d_offsets, n_rec, nullptr, nullptr, d_match_offsets, 0)) return rc;
  } else {
    if (fast) batch_iter_fast<0><<<grid, 512, fsm, st>>>(a);
    else batch_iter<0><<<grid, 256, 0, st>>>(a);
    RB_LAUNCH_CHECK("batch_iter<0>");
  }
  // ---- exclusive scan over n_rec + 1 entries ----
  unsigned long long* grand;
  if (int rc = prefix_sum(d_match_offsets, d_match_offsets, n_rec + 1, &grand)) return rc;
  uint64_t* h = &h_scalars_->iter_total;
  if (grow) {  // every span, into a buffer sized by the count
    RB_CUDA(cudaMemcpyAsync(h, grand, 8, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    a.out_spans = (uint64_t*)grow->ensure(std::max<uint64_t>(*h, 1) * 16);
    if (!a.out_spans) return fail("out of device memory (batch spans)");
    a.cap = *h;
  }
  // ---- write ----
  if (a.cap > 0 && cand) {
    if (int rc = cand_batch(3, d_text, d_offsets, n_rec, nullptr, a.out_spans, d_match_offsets, a.cap)) return rc;
  } else if (a.cap > 0) {
    a.fwd_only = 0;
    if (fast) batch_iter_fast<1><<<grid, 512, fsm, st>>>(a);
    else batch_iter<1><<<grid, 256, 0, st>>>(a);
    RB_LAUNCH_CHECK("batch_iter<1>");
  }
  RB_CUDA(cudaMemcpyAsync(h, grand, 8, cudaMemcpyDeviceToHost, st));
  RB_CUDA(cudaStreamSynchronize(st));
  *total = *h;
  return 0;
}

// Regex::captures per record: the first match of every record (find_batch), then the Pike VM over the
// record-relative window of each (kernels.cu pike_captures with rec_offsets).
int Regex::captures_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_slots, uint32_t* d_bits) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (int rc = ensure_capture_program()) return rc;
  if (n_rec == 0) return 0;
  uint64_t* d_spans = (uint64_t*)cap_span_.ensure(n_rec * 16);
  if (!d_spans) return fail("out of device memory (captures)");
  if (int rc = find_batch_device(d_text, d_offsets, n_rec, d_spans, d_bits)) return rc;
  if (int rc = launch_captures(d_text, 0, d_spans, n_rec, d_slots, d_offsets, d_bits)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  // exec.rs:896-906: a record matches when the NFA found group 0 in its window
  slot_found_bits<<<(uint32_t)((n_rec + 255) / 256), 256, 0, st>>>(d_slots, 2 * (uint32_t)n_groups_, n_rec, d_bits);
  RB_LAUNCH_CHECK("slot_found_bits");
  RB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int Regex::set_matches_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_masks) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (n_rec == 0) return 0;
  const uint32_t mw = (uint32_t)std::max<size_t>(1, (patterns_.size() + 63) / 64);
  if (patterns_.empty()) {
    if (int rc = init_device()) return rc;
    RB_CUDA(cudaMemsetAsync(d_masks, 0, n_rec * 8 * mw, (cudaStream_t)stream_));
    RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    return 0;
  }
  if (!groups_.empty()) return set_matches_batch_grouped(d_text, d_offsets, n_rec, d_masks);
  stats.groups = 1;
  DeviceDfa* fwd;
  if (int rc = ensure(kFwdUnanchoredAll, &fwd)) return rc;
  BatchArgs a{};
  size_t smem;
  uint32_t per_sm;
  batch_args(&a, d_text, d_offsets, n_rec, fwd, nullptr, 0, 0, &smem, &per_sm);
  a.out_masks = d_masks;
  RB_CUDA(allow_smem(set_matches_batch, smem));
  set_matches_batch<<<(uint32_t)((n_rec + 255) / 256), 256, smem, (cudaStream_t)stream_>>>(a);
  RB_LAUNCH_CHECK("set_matches_batch");
  RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  return 0;
}

// One launch for every group of a grouped set (gridDim.y = groups): each CTA stages its group's table when it fits.
int Regex::set_matches_batch_grouped(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_masks) {
  if (int rc = init_device()) return rc;
  const uint32_t n_pat = (uint32_t)patterns_.size(), n_g = (uint32_t)groups_.size(), rw = (n_pat + 63) / 64;
  cudaStream_t st = (cudaStream_t)stream_;
  std::vector<GroupDesc> descs(n_g);
  size_t smem = 0;
  for (uint32_t g = 0; g < n_g; g++) {
    Regex* gr = groups_[g].get();
    gr->tuning = tuning;
    gr->set_stream(stream_);
    DeviceDfa* fwd;
    if (gr->ensure(kFwdUnanchoredAll, &fwd)) return fail(gr->last_error());
    const size_t s = smem_for(fwd->view);
    descs[g].view = fwd->view;
    descs[g].lo = group_first_[g];
    descs[g].hi = g + 1 < n_g ? group_first_[g + 1] : n_pat;
    descs[g].use_smem = s != 0;
    smem = std::max(smem, s);
  }
  GroupDesc* d_descs = (GroupDesc*)group_descs_.ensure(n_g * sizeof(GroupDesc));
  if (!d_descs) return fail("out of device memory (group tables)");
  RB_CUDA(cudaMemcpyAsync(d_descs, descs.data(), n_g * sizeof(GroupDesc), cudaMemcpyHostToDevice, st));
  RB_CUDA(cudaMemsetAsync(d_masks, 0, n_rec * 8 * rw, st));
  GroupBatchArgs a{};
  a.groups = d_descs;
  a.text = d_text;
  a.offsets = d_offsets;
  a.n_rec = n_rec;
  a.out_masks = d_masks;
  a.row_words = rw;
  a.n_patterns = n_pat;
  RB_CUDA(allow_smem(set_matches_batch_groups, smem));
  set_matches_batch_groups<<<dim3((uint32_t)((n_rec + 255) / 256), n_g), 256, smem, st>>>(a);
  RB_LAUNCH_CHECK("set_matches_batch_groups");
  RB_CUDA(cudaStreamSynchronize(st));
  stats.groups = n_g;
  return 0;
}

// exclusive prefix sum of in[0, n) into out (kernels.cu scan_counts_local / scan_block_sums / scan_add_block_offsets)
int Regex::prefix_sum(const uint64_t* in, uint64_t* out, uint64_t n, unsigned long long** d_total) {
  cudaStream_t st = (cudaStream_t)stream_;
  const uint64_t n_blocks = (n + 1023) / 1024;
  uint64_t* block_sums = (uint64_t*)block_sums_.ensure((n_blocks + 1) * 8);
  if (!block_sums) return fail("out of device memory (scan)");
  *d_total = (unsigned long long*)(block_sums + n_blocks);
  if (n_blocks == 0) {
    RB_CUDA(cudaMemsetAsync(*d_total, 0, 8, st));
    return 0;
  }
  scan_counts_local<<<(uint32_t)n_blocks, 1024, 0, st>>>(in, out, block_sums, n);
  RB_LAUNCH_CHECK("scan_counts_local");
  scan_block_sums<<<1, 1024, 0, st>>>(block_sums, n_blocks, *d_total);
  RB_LAUNCH_CHECK("scan_block_sums");
  scan_add_block_offsets<<<(uint32_t)n_blocks, 1024, 0, st>>>(out, block_sums, n);
  RB_LAUNCH_CHECK("scan_add_block_offsets");
  return 0;
}

// ------------------------------------------------------- replace_all / split ----
// All spans of the haystack in spans_all_ (device); *m = their number.
int Regex::all_spans_device(const uint8_t* d_text, uint64_t n, uint64_t** d_spans, uint64_t* m) {
  uint64_t total = 0;
  if (int rc = find_all_device(d_text, n, 0, nullptr, 0, &total)) return rc;
  uint64_t* sp = (uint64_t*)spans_all_.ensure(std::max<uint64_t>(total, 1) * 16);
  if (!sp) return fail("out of device memory (spans)");
  if (total) {
    uint64_t again = 0;
    if (int rc = find_all_device(d_text, n, 0, sp, total, &again)) return rc;
  }
  *d_spans = sp;
  *m = total;
  return 0;
}

int Regex::replace_device(const uint8_t* d_text, uint64_t n, const uint8_t* rep, uint64_t rep_len, bool expand, uint64_t limit,
                          uint8_t* d_out, uint64_t out_cap, uint64_t* out_len) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (int rc = replace_prepare(d_text, n, rep, rep_len, expand, limit, out_len)) return rc;
  if (!d_out) return 0;
  return replace_emit(d_out, out_cap);
}

// Template, spans and prefix sums of one replace call; leaves everything replace_emit needs in
// rep_args_ / rep_lits_ and the device scratch.
int Regex::replace_prepare(const uint8_t* d_text, uint64_t n, const uint8_t* rep, uint64_t rep_len, bool expand, uint64_t limit,
                           uint64_t* out_len) {
  if (is_set_) return fail("replace requires exactly one pattern");
  bool needs_groups = false;
  if (int rc = replace_template(rep, rep_len, expand, &needs_groups)) return rc;
  uint64_t* spans;
  uint64_t m;
  if (int rc = all_spans_device(d_text, n, &spans, &m)) return rc;
  if (limit && m > limit) m = limit;
  uint64_t* d_slots = nullptr;
  if (needs_groups && m) {  // `$1`, `$name`: the groups of every match (capture pass on the narrowed windows)
    d_slots = (uint64_t*)cap_slots_.ensure(m * 2 * (uint64_t)n_groups_ * 8);
    if (!d_slots) return fail("out of device memory (captures)");
    if (int rc = captures_device(d_text, n, spans, m, d_slots)) return rc;
  }
  return replace_sums(d_text, n, spans, m, d_slots, out_len);
}

// ---- the replacement template (src/expand.rs:50-90) ----
int Regex::replace_template(const uint8_t* rep, uint64_t rep_len, bool expand, bool* needs_groups_out) {
  rep_args_.assign(sizeof(ReplaceArgs), 0);
  ReplaceArgs& a = *reinterpret_cast<ReplaceArgs*>(rep_args_.data());
  a = ReplaceArgs{};
  std::vector<uint8_t>& lits = rep_lits_;
  lits.clear();
  auto literal = [&](const uint8_t* p, uint64_t len) -> bool {
    if (len == 0) return true;
    if (a.n_parts && !(a.part_len[a.n_parts - 1] & kRepGroup) && a.part_off[a.n_parts - 1] + a.part_len[a.n_parts - 1] == lits.size()) {
      a.part_len[a.n_parts - 1] += (uint32_t)len;  // extend the previous literal part
    } else {
      if (a.n_parts == kMaxRepParts) return false;
      a.part_off[a.n_parts] = (uint32_t)lits.size();
      a.part_len[a.n_parts++] = (uint32_t)len;
    }
    lits.insert(lits.end(), p, p + len);
    a.lit_total += len;
    return true;
  };
  bool fits = true, needs_groups = false;
  if (!expand) {
    fits = literal(rep, rep_len);
  } else {
    uint64_t i = 0;
    auto cap_letter = [](uint8_t b) { return (b >= '0' && b <= '9') || (b >= 'a' && b <= 'z') || (b >= 'A' && b <= 'Z') || b == '_'; };
    while (i < rep_len && fits) {
      uint64_t j = i;
      while (j < rep_len && rep[j] != '$') j++;
      fits = literal(rep + i, j - i);
      i = j;
      if (i >= rep_len) break;
      if (i + 1 < rep_len && rep[i + 1] == '$') { fits = fits && literal(rep + i, 1); i += 2; continue; }
      // find_cap_ref (expand.rs:128-167)
      uint64_t k = i + 1;
      bool brace = false;
      if (k < rep_len && rep[k] == '{') { brace = true; k++; }
      uint64_t ce = k;
      while (ce < rep_len && cap_letter(rep[ce])) ce++;
      bool ok = rep_len - i > 1 && ce > k;
      std::string name;
      if (ok) {
        name.assign((const char*)rep + k, ce - k);
        if (brace) { if (ce < rep_len && rep[ce] == '}') ce++; else ok = false; }
      }
      if (!ok) { fits = fits && literal(rep + i, 1); i += 1; continue; }  // a lone '$'
      i = ce;
      // expand.rs:78-87: a number is a group index, anything else a group name; a group the pattern
      // does not have expands to nothing
      long g = -1;
      if (name.find_first_not_of("0123456789") == std::string::npos) {
        g = name.size() <= 9 ? std::atol(name.c_str()) : -1;
      } else {
        for (const auto& gn : group_name_index_) if (gn.first == name) g = gn.second;
      }
      if (g >= 0 && g < n_groups_) {
        if (a.n_parts == kMaxRepParts) { fits = false; break; }
        a.part_len[a.n_parts] = kRepGroup | (uint32_t)g;
        a.part_off[a.n_parts++] = 0;
        if (g > 0) needs_groups = true;
      }
    }
  }
  if (!fits) return fail("replacement template has too many parts");
  *needs_groups_out = needs_groups;
  return 0;
}

int Regex::replace_sums(const uint8_t* d_text, uint64_t n, const uint64_t* spans, uint64_t m, const uint64_t* slots, uint64_t* out_len) {
  ReplaceArgs& a = *reinterpret_cast<ReplaceArgs*>(rep_args_.data());
  const std::vector<uint8_t>& lits = rep_lits_;
  cudaStream_t st = (cudaStream_t)stream_;
  uint64_t* lens = (uint64_t*)lens_.ensure(std::max<uint64_t>(m, 1) * 8);
  uint64_t* before = (uint64_t*)lens_before_.ensure(std::max<uint64_t>(m, 1) * 8);
  uint8_t* d_lits = (uint8_t*)lits_.ensure(std::max<size_t>(lits.size(), 16));
  if (!lens || !before || !d_lits) return fail("out of device memory (replace scratch)");
  uint64_t* reps_before = (uint64_t*)reps_before_.ensure(std::max<uint64_t>(m, 1) * 8);
  if (!reps_before) return fail("out of device memory (replace scratch)");
  a.text = d_text;
  a.n = n;
  a.spans = spans;
  a.n_matches = m;
  a.lens_before = before;
  a.reps_before = reps_before;
  a.lits = d_lits;
  a.slots = slots;
  a.n_slots = slots ? 2 * (uint32_t)n_groups_ : 0;
  uint64_t matched = 0, replaced = 0;
  if (m) {
    auto prefix = [&](uint64_t* out, uint64_t* total) -> int {  // exclusive prefix sum of lens[] into out[]
      unsigned long long* grand;
      if (int rc = prefix_sum(lens, out, m, &grand)) return rc;
      RB_CUDA(d2h(total, grand, 8));
      return 0;
    };
    span_lengths<<<grid_for(m, 256, 8), 256, 0, st>>>(spans, m, lens);
    RB_LAUNCH_CHECK("span_lengths");
    if (int rc = prefix(before, &matched)) return rc;
    replace_lengths<<<grid_for(m, 256, 8), 256, 0, st>>>(a, lens);
    RB_LAUNCH_CHECK("replace_lengths");
    if (int rc = prefix(reps_before, &replaced)) return rc;
  }
  rep_totals_[0] = matched;
  rep_totals_[1] = replaced;
  *out_len = n - matched + replaced;
  return 0;
}

int Regex::replace_emit(uint8_t* d_out, uint64_t out_cap) {
  ReplaceArgs a = *reinterpret_cast<ReplaceArgs*>(rep_args_.data());
  const std::vector<uint8_t>& lits = rep_lits_;
  cudaStream_t st = (cudaStream_t)stream_;
  uint8_t* d_lits = (uint8_t*)lits_.ptr;
  const uint64_t n = a.n, m = a.n_matches;
  if (!lits.empty()) RB_CUDA(cudaMemcpyAsync(d_lits, lits.data(), lits.size(), cudaMemcpyHostToDevice, st));
  a.out = d_out;
  a.out_cap = out_cap;
  if (n) {
    replace_gaps<<<grid_for(((n + 2047) / 2048) * 32, 256, 8), 256, 0, st>>>(a, rep_totals_[0], rep_totals_[1]);
    RB_LAUNCH_CHECK("replace_gaps");
  }
  if (m && a.n_parts) {
    replace_matches<<<grid_for(m * 32, 256, 8), 256, 0, st>>>(a);
    RB_LAUNCH_CHECK("replace_matches");
  }
  RB_CUDA(cudaStreamSynchronize(st));  // `lits` and the caller's buffers may go away now
  return 0;
}

int Regex::replace_host(const uint8_t* text, uint64_t n, const uint8_t* rep, uint64_t rep_len, bool expand, uint64_t limit, uint8_t* out,
                        uint64_t out_cap, uint64_t* out_len) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  int rc;
  const uint8_t* d = upload_text(text, n, &rc);
  if (rc) return rc;
  if ((rc = replace_prepare(d, n, rep, rep_len, expand, limit, out_len))) return rc;
  if (!out) return 0;
  uint8_t* d_out = (uint8_t*)rep_out_.ensure(std::max<uint64_t>(*out_len, 16));
  if (!d_out) return fail("out of device memory (replace output)");
  if ((rc = replace_emit(d_out, *out_len))) return rc;
  const uint64_t k = std::min(out_cap, *out_len);
  if (k) RB_CUDA(d2h(out, d_out, k));
  return 0;
}

int Regex::split_device(const uint8_t* d_text, uint64_t n, bool has_limit, uint64_t limit, uint64_t* d_pieces, uint64_t cap, uint64_t* n_pieces) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *n_pieces = 0;
  if (is_set_) return fail("split requires exactly one pattern");
  if (has_limit && limit == 0) return 0;  // re_bytes.rs:738-740
  uint64_t* spans;
  uint64_t m;
  if (int rc = all_spans_device(d_text, n, &spans, &m)) return rc;
  uint64_t last_end = 0;
  if (m) RB_CUDA(d2h(&last_end, spans + 2 * m - 1, 8));
  // Split yields one piece per match and the rest of the text when it is not empty (re_bytes.rs:702-720)
  const uint64_t p_split = m + (last_end < n ? 1 : 0);
  uint64_t pieces = p_split;
  int last_is_rest = 0;
  if (has_limit && p_split >= limit - 1) {  // SplitN: the limit-th piece is whatever remains, empty or not (re_bytes.rs:737-748)
    pieces = limit;
    last_is_rest = 1;
  }
  *n_pieces = pieces;
  if (d_pieces && pieces && cap) {
    split_pieces<<<grid_for(pieces, 256, 8), 256, 0, (cudaStream_t)stream_>>>(spans, m, n, pieces, last_is_rest, d_pieces, cap);
    RB_LAUNCH_CHECK("split_pieces");
    RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  }
  return 0;
}

int Regex::split_host(const uint8_t* text, uint64_t n, bool has_limit, uint64_t limit, uint64_t* pieces, uint64_t cap, uint64_t* n_pieces) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  int rc;
  const uint8_t* d = upload_text(text, n, &rc);
  if (rc) return rc;
  if ((rc = split_device(d, n, has_limit, limit, nullptr, 0, n_pieces))) return rc;
  if (!pieces || !cap || !*n_pieces) return 0;
  const uint64_t k = std::min(cap, *n_pieces);
  uint64_t* d_p = (uint64_t*)pieces_.ensure(k * 16);
  if (!d_p) return fail("out of device memory (pieces)");
  if ((rc = split_device(d, n, has_limit, limit, d_p, k, n_pieces))) return rc;
  RB_CUDA(d2h(pieces, d_p, k * 16));
  return 0;
}

// ------------------------------------------------------------ capture groups ----
int Regex::ensure_capture_program() {
  if (cap_n_insts_) return 0;
  if (is_set_ || patterns_.size() != 1) return fail("captures require exactly one pattern (exec.rs:587-589)");
  if (int rc = init_device()) return rc;
  rb::CompileOptions co;
  co.only_utf8 = opt_.only_utf8;
  co.size_limit = opt_.size_limit;
  co.unanchored_prefix = true;
  co.saves = true;
  rb::Program prog;
  rb::Error err;
  if (!rb::compile(exprs_, co, &prog, &err)) return fail(err.msg);
  std::vector<NfaInst> insts(prog.insts.size());
  for (size_t i = 0; i < insts.size(); i++) {
    const rb::Inst& in = prog.insts[i];
    insts[i].op_look_lo_hi = (uint32_t)in.op | ((uint32_t)in.look << 8) | ((uint32_t)in.lo << 16) | ((uint32_t)in.hi << 24);
    insts[i].a = in.a;
    insts[i].b = in.b;
  }
  NfaInst* d = (NfaInst*)cap_insts_.ensure(insts.size() * sizeof(NfaInst));
  if (!d) return fail("out of device memory (capture program)");
  RB_CUDA(cudaMemcpyAsync(d, insts.data(), insts.size() * sizeof(NfaInst), cudaMemcpyHostToDevice, (cudaStream_t)stream_));
  RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  cap_n_insts_ = (uint32_t)insts.size();
  cap_start_ = prog.start;
  cap_anchored_ = prog.is_anchored_start;
  return 0;
}

int Regex::captures_device(const uint8_t* d_text, uint64_t n, const uint64_t* d_spans, uint64_t m, uint64_t* d_slots) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  if (int rc = ensure_capture_program()) return rc;
  if (m == 0) return 0;
  if (int rc = launch_captures(d_text, n, d_spans, m, d_slots, nullptr, nullptr)) return rc;
  RB_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
  return 0;
}

// pike_captures over m spans (rec_offsets / rec_found: batched records, see launch.h CapArgs)
int Regex::launch_captures(const uint8_t* d_text, uint64_t n, const uint64_t* d_spans, uint64_t m, uint64_t* d_slots,
                           const uint64_t* rec_offsets, const uint32_t* rec_found, const uint64_t* rec_csr, uint64_t n_rec) {
  CapArgs a{};
  a.insts = (const NfaInst*)cap_insts_.ptr;
  a.n_insts = cap_n_insts_;
  a.start_ip = cap_start_;
  a.anchored_start = cap_anchored_ ? 1 : 0;
  a.n_slots = 2 * (uint32_t)n_groups_;
  a.text = d_text;
  a.n = n;
  a.spans = d_spans;
  a.n_matches = m;
  a.slots = d_slots;
  // kernels.cu pike_captures: two slot tables, thread caps, stack positions, four index arrays, stack tags
  const uint64_t ni = a.n_insts, ns = a.n_slots;
  a.per_thread = (2 * ni * ns * 8 + ns * 8 + (2 * ni + 4) * 8 + 4 * ni * 4 + (2 * ni + 4) * 4 + 15) / 16 * 16;
  if (a.per_thread > (8u << 20)) return fail("the pattern is too large for capture extraction on the device (program x groups)");
  uint64_t threads = std::min<uint64_t>((m + 63) / 64 * 64, 16384);
  while (threads > 64 && threads * a.per_thread > (1ull << 30)) threads /= 2;
  a.scratch = (uint8_t*)cap_scratch_.ensure(threads * a.per_thread);
  if (!a.scratch) return fail("out of device memory (capture scratch)");
  a.rec_offsets = rec_offsets;
  a.rec_found = rec_found;
  a.rec_csr = rec_csr;
  a.n_rec = n_rec;
  pike_captures<<<(uint32_t)(threads / 64), 64, 0, (cudaStream_t)stream_>>>(a);
  RB_LAUNCH_CHECK("pike_captures");
  return 0;
}

int Regex::captures_at_host(const uint8_t* text, uint64_t n, uint64_t start, bool* found, uint64_t* slots) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  uint64_t s = 0, e = 0;
  if (int rc = find_at_host(text, n, start, found, &s, &e)) return rc;  // the DFA path finds the match (exec.rs:547-556)
  if (!*found) return 0;
  // the window the capture pass reads: one byte of look-behind, two characters of look-ahead
  uint8_t* d = (uint8_t*)text_.ensure(n + 64);
  const uint64_t lo = s ? s - 1 : 0, hi = std::min<uint64_t>(n, e + 8);
  cudaStream_t st = (cudaStream_t)stream_;
  RB_CUDA(cudaMemcpyAsync(d + lo, text + lo, hi - lo, cudaMemcpyHostToDevice, st));
  uint64_t* d_span = (uint64_t*)cap_span_.ensure(16);
  const uint32_t ns = 2 * (uint32_t)n_groups_;
  uint64_t* d_slots = (uint64_t*)cap_slots_.ensure(ns * 8);
  if (!d_span || !d_slots) return fail("out of device memory (captures)");
  const uint64_t span[2] = {s, e};
  RB_CUDA(cudaMemcpyAsync(d_span, span, 16, cudaMemcpyHostToDevice, st));
  RB_CUDA(cudaStreamSynchronize(st));
  if (int rc = captures_device(d, hi, d_span, 1, d_slots)) return rc;  // (hi bounds a window the pass never leaves)
  RB_CUDA(d2h(slots, d_slots, ns * 8));
  *found = slots[0] != kNone;  // exec.rs:896-906: the result is what the NFA found in the window
  return 0;
}

int Regex::captures_all_host(const uint8_t* text, uint64_t n, uint64_t* slots, uint64_t cap, uint64_t* m) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  int rc;
  const uint8_t* d = upload_text(text, n, &rc);
  if (rc) return rc;
  uint64_t* spans;
  if ((rc = all_spans_device(d, n, &spans, m))) return rc;
  const uint64_t k = std::min(cap, *m);
  if (!slots || !k) return 0;
  const uint32_t ns = 2 * (uint32_t)n_groups_;
  uint64_t* d_slots = (uint64_t*)cap_slots_.ensure(k * ns * 8);
  if (!d_slots) return fail("out of device memory (captures)");
  if ((rc = captures_device(d, n, spans, k, d_slots))) return rc;
  RB_CUDA(d2h(slots, d_slots, k * ns * 8));
  // CaptureMatches (re_trait.rs:236-263) iterates on what read_captures_at returns, i.e. on the NFA's
  // group 0.  That is the find_iter span except where the reverse-on-slice quirk (SURVEY H1) gave
  // the DFA a start no match begins at; from the first such match on, iterate like the reference.
  std::vector<uint64_t> h_spans(2 * k);
  RB_CUDA(d2h(h_spans.data(), spans, k * 16));
  uint64_t j = 0;
  while (j < k && slots[j * ns] == h_spans[2 * j] && slots[j * ns + 1] == h_spans[2 * j + 1]) j++;
  if (j == k && *m <= cap) return 0;
  if (j == k) return 0;  // the caller's buffer ends before any divergence
  auto next_after_empty = [&](uint64_t i) -> uint64_t {  // exec.rs:335-337, 375-377
    if (!only_utf8 || i >= n) return i + 1;
    const uint8_t b = text[i];
    return i + (b <= 0x7F ? 1 : b <= 0xDF ? 2 : b <= 0xEF ? 3 : 4);
  };
  uint64_t last_end = 0, last_match = kNone;
  if (j) {
    const uint64_t ps = h_spans[2 * (j - 1)], pe = h_spans[2 * (j - 1) + 1];
    last_end = ps == pe ? next_after_empty(pe) : pe;
    last_match = pe;
  }
  std::vector<uint64_t> one(ns);
  uint64_t count = j;
  while (last_end <= n) {
    bool found = false;
    if ((rc = captures_at_host(text, n, last_end, &found, one.data()))) return rc;
    if (!found) break;
    const uint64_t s = one[0], e = one[1];
    if (s == e) {
      last_end = next_after_empty(e);
      if (e == last_match) continue;
    } else {
      last_end = e;
    }
    last_match = e;
    if (count < cap) std::copy(one.begin(), one.end(), slots + count * ns);
    count++;
  }
  *m = count;
  return 0;
}

// ------------------------------------------- batched records: replacen / splitn / captures_iter ----
// Each record is its own haystack.  The spans come from the per-record find_iter (iter_batch: record-relative,
// CSR-shaped, in bspans_ / bmoff_).  Replace makes them relative to offsets[0] and runs the whole-haystack
// kernels unchanged on the concatenated records; split and captures find each item's record by a binary search.
int Regex::replace_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, const uint8_t* rep, uint64_t rep_len,
                                bool expand, uint64_t limit, uint64_t* d_out_offsets, uint8_t* d_out, uint64_t out_cap, uint64_t* out_len) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *out_len = 0;
  if (is_set_) return fail("replace requires exactly one pattern");
  bool needs_groups = false;
  if (int rc = replace_template(rep, rep_len, expand, &needs_groups)) return rc;
  if (needs_groups)
    if (int rc = ensure_capture_program()) return rc;
  uint64_t* moff = (uint64_t*)bmoff_.ensure((n_rec + 1) * 8);
  if (!moff) return fail("out of device memory (batch)");
  uint64_t m = 0;
  if (int rc = iter_batch(d_text, d_offsets, n_rec, moff, nullptr, 0, &m, &bspans_)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_rec == 0) {
    RB_CUDA(cudaMemsetAsync(d_out_offsets, 0, 8, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  uint64_t* spans = (uint64_t*)bspans_.ptr;
  if (limit && m > limit) {  // replacen: the first `limit` matches of every record
    uint64_t* koff = (uint64_t*)bkoff_.ensure((n_rec + 1) * 8);
    if (!koff) return fail("out of device memory (batch)");
    csr_counts<<<grid_for(n_rec + 1, 256, 8), 256, 0, st>>>(moff, n_rec, limit, koff);
    RB_LAUNCH_CHECK("csr_counts");
    unsigned long long* grand;
    if (int rc = prefix_sum(koff, koff, n_rec + 1, &grand)) return rc;
    uint64_t kept = 0;
    RB_CUDA(d2h(&kept, grand, 8));
    if (kept < m) {
      uint64_t* ks = (uint64_t*)bkspans_.ensure(std::max<uint64_t>(kept, 1) * 16);
      if (!ks) return fail("out of device memory (batch spans)");
      batch_keep_spans<<<grid_for(m, 256, 8), 256, 0, st>>>(moff, koff, n_rec, spans, m, ks);
      RB_LAUNCH_CHECK("batch_keep_spans");
      spans = ks;
      moff = koff;
      m = kept;
    }
  }
  uint64_t first = 0, last = 0;
  RB_CUDA(d2h(&first, d_offsets, 8));
  RB_CUDA(d2h(&last, d_offsets + n_rec, 8));
  const uint32_t ns = 2 * (uint32_t)n_groups_;
  uint64_t* slots = nullptr;
  if (needs_groups && m) {  // record-relative groups of every kept match, the window cut at its record's end
    slots = (uint64_t*)bslots_.ensure(m * ns * 8);
    if (!slots) return fail("out of device memory (captures)");
    if (int rc = launch_captures(d_text, 0, spans, m, slots, d_offsets, nullptr, moff, n_rec)) return rc;
  }
  if (m) {
    batch_to_base<<<grid_for(m, 256, 8), 256, 0, st>>>(d_offsets, moff, n_rec, spans, m, slots, ns);
    RB_LAUNCH_CHECK("batch_to_base");
  }
  if (int rc = replace_sums(d_text + first, last - first, spans, m, slots, out_len)) return rc;
  const ReplaceArgs& ra = *reinterpret_cast<const ReplaceArgs*>(rep_args_.data());
  batch_replace_offsets<<<grid_for(n_rec + 1, 256, 8), 256, 0, st>>>(d_offsets, moff, n_rec, ra.lens_before, ra.reps_before, m, rep_totals_[0],
                                                                      rep_totals_[1], d_out_offsets);
  RB_LAUNCH_CHECK("batch_replace_offsets");
  if (!d_out) {
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  return replace_emit(d_out, out_cap);
}

int Regex::split_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, bool has_limit, uint64_t limit,
                              uint64_t* d_piece_offsets, uint64_t* d_pieces, uint64_t cap, uint64_t* n_total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *n_total = 0;
  if (is_set_) return fail("split requires exactly one pattern");
  if (int rc = init_device()) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_rec == 0 || (has_limit && limit == 0)) {  // re_bytes.rs:738-740: splitn(0) yields nothing
    RB_CUDA(cudaMemsetAsync(d_piece_offsets, 0, (n_rec + 1) * 8, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  uint64_t* moff = (uint64_t*)bmoff_.ensure((n_rec + 1) * 8);
  if (!moff) return fail("out of device memory (batch)");
  uint64_t m = 0;
  if (int rc = iter_batch(d_text, d_offsets, n_rec, moff, nullptr, 0, &m, &bspans_)) return rc;
  const uint64_t* spans = (const uint64_t*)bspans_.ptr;
  batch_split_counts<<<grid_for(n_rec + 1, 256, 8), 256, 0, st>>>(d_offsets, moff, spans, n_rec, has_limit ? 1 : 0, limit, d_piece_offsets);
  RB_LAUNCH_CHECK("batch_split_counts");
  unsigned long long* grand;
  if (int rc = prefix_sum(d_piece_offsets, d_piece_offsets, n_rec + 1, &grand)) return rc;
  RB_CUDA(d2h(n_total, grand, 8));
  const uint64_t k = d_pieces ? std::min(cap, *n_total) : 0;
  if (k) {
    batch_split_pieces<<<grid_for(k, 256, 8), 256, 0, st>>>(d_offsets, moff, spans, d_piece_offsets, n_rec, has_limit ? 1 : 0, limit,
                                                            d_pieces, k);
    RB_LAUNCH_CHECK("batch_split_pieces");
  }
  RB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int Regex::captures_iter_batch_device(const uint8_t* d_text, const uint64_t* d_offsets, uint64_t n_rec, uint64_t* d_match_offsets,
                                      uint64_t* d_slots, uint64_t cap, uint64_t* n_total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *n_total = 0;
  if (int rc = ensure_capture_program()) return rc;
  if (!d_slots) cap = 0;
  uint64_t* moff = (uint64_t*)bmoff_.ensure((n_rec + 1) * 8);
  if (!moff) return fail("out of device memory (batch)");
  uint64_t m = 0;
  if (int rc = iter_batch(d_text, d_offsets, n_rec, moff, nullptr, 0, &m, &bspans_)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_rec == 0) {
    RB_CUDA(cudaMemsetAsync(d_match_offsets, 0, 8, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  const uint32_t ns = 2 * (uint32_t)n_groups_;
  const uint64_t* spans = (const uint64_t*)bspans_.ptr;
  const uint64_t words = (n_rec + 31) / 32;
  uint64_t* slots = (uint64_t*)bslots_.ensure(std::max<uint64_t>(m, 1) * ns * 8);
  uint32_t* flags = (uint32_t*)bflags_.ensure((words + 1) * 4);
  uint64_t* list = (uint64_t*)blist_.ensure(n_rec * 8);
  if (!slots || !flags || !list) return fail("out of device memory (captures)");
  unsigned int* n_list = (unsigned int*)(flags + words);
  RB_CUDA(cudaMemsetAsync(flags, 0, (words + 1) * 4, st));
  if (m) {
    if (int rc = launch_captures(d_text, 0, spans, m, slots, d_offsets, nullptr, moff, n_rec)) return rc;
    batch_diverged<<<(uint32_t)((m + 255) / 256), 256, 0, st>>>(moff, n_rec, spans, m, slots, ns, flags, list, n_list);
    RB_LAUNCH_CHECK("batch_diverged");
  }
  unsigned int n_redo = 0;
  RB_CUDA(d2h(&n_redo, n_list, 4));
  if (n_redo == 0) {  // group 0 is the find_iter span everywhere (always so without look-around): the CSR stands
    RB_CUDA(cudaMemcpyAsync(d_match_offsets, moff, (n_rec + 1) * 8, cudaMemcpyDeviceToDevice, st));
    if (std::min(cap, m)) RB_CUDA(cudaMemcpyAsync(d_slots, slots, std::min(cap, m) * ns * 8, cudaMemcpyDeviceToDevice, st));
    RB_CUDA(cudaStreamSynchronize(st));
    *n_total = m;
    return 0;
  }
  // CaptureMatches (re_trait.rs:236-263) iterates on the NFA's group 0.  Where that differs from the find_iter span
  // (the reverse-on-slice rule, SURVEY H1), captures_all_host, which follows the reference from the first such
  // match on, reruns the record alone.  Such records are rare, so this path is driven from the host.  Everything
  // it needs of d_text and d_offsets is read first: captures_all_host reuses the whole-haystack scratch.
  std::vector<uint64_t> recs(n_redo);
  RB_CUDA(d2h(recs.data(), list, n_redo * 8));
  std::vector<std::vector<uint8_t>> bytes(n_redo);
  for (unsigned int i = 0; i < n_redo; i++) {
    uint64_t lohi[2];
    RB_CUDA(d2h(lohi, d_offsets + recs[i], 16));
    bytes[i].resize(lohi[1] - lohi[0]);
    if (!bytes[i].empty()) RB_CUDA(d2h(bytes[i].data(), d_text + lohi[0], bytes[i].size()));
  }
  std::vector<std::vector<uint64_t>> rows(n_redo);
  std::vector<uint64_t> counts(n_redo);
  for (unsigned int i = 0; i < n_redo; i++) {
    const uint64_t len = bytes[i].size(), room = len + 2;  // a record of len bytes has at most len + 1 matches
    rows[i].resize(room * ns);
    if (int rc = captures_all_host(bytes[i].data(), len, rows[i].data(), room, &counts[i])) return rc;
  }
  // the new CSR: the old counts with the redone ones, scanned; old rows move, redone rows are uploaded
  uint64_t* cnt = (uint64_t*)bkoff_.ensure((n_rec + 1) * 8);
  if (!cnt) return fail("out of device memory (batch)");
  csr_counts<<<grid_for(n_rec + 1, 256, 8), 256, 0, st>>>(moff, n_rec, kNone, cnt);
  RB_LAUNCH_CHECK("csr_counts");
  for (unsigned int i = 0; i < n_redo; i++) RB_CUDA(cudaMemcpyAsync(cnt + recs[i], &counts[i], 8, cudaMemcpyHostToDevice, st));
  unsigned long long* grand;
  if (int rc = prefix_sum(cnt, d_match_offsets, n_rec + 1, &grand)) return rc;
  RB_CUDA(d2h(n_total, grand, 8));
  if (cap) {
    batch_move_rows<<<grid_for(m, 256, 8), 256, 0, st>>>(moff, d_match_offsets, n_rec, flags, slots, m, ns, d_slots, cap);
    RB_LAUNCH_CHECK("batch_move_rows");
    for (unsigned int i = 0; i < n_redo; i++) {
      uint64_t at = 0;
      RB_CUDA(d2h(&at, d_match_offsets + recs[i], 8));
      const uint64_t k = at < cap ? std::min(counts[i], cap - at) : 0;
      if (k) RB_CUDA(cudaMemcpyAsync(d_slots + at * ns, rows[i].data(), k * ns * 8, cudaMemcpyHostToDevice, st));
    }
  }
  RB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------ host wrappers ----
// device -> host on the library's stream, complete on return
int Regex::d2h(void* dst, const void* src, size_t bytes) {
  int e = (int)cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream_);
  if (e != cudaSuccess) return e;
  return (int)cudaStreamSynchronize((cudaStream_t)stream_);
}

const uint8_t* Regex::upload_text(const uint8_t* text, uint64_t n, int* rc) {
  if ((*rc = init_device())) return nullptr;
  uint8_t* d = (uint8_t*)text_.ensure(n + 64);
  if (!d) { *rc = fail("out of device memory (haystack)"); return nullptr; }
  if (n) {  // stream-ordered with the kernels that read it
    int e = (int)cudaMemcpyAsync(d, text, n, cudaMemcpyHostToDevice, (cudaStream_t)stream_);
    if (e != cudaSuccess) { *rc = check(e, "haystack upload"); return nullptr; }
  }
  return d;
}

int Regex::side_streams() {
  if (copy_stream_) return 0;
  cudaStream_t s1, s2;
  RB_CUDA(cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking));
  RB_CUDA(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
  copy_stream_ = s1;
  back_stream_ = s2;
  return 0;
}

// Bytes per uploaded piece of a pipelined host find_all (RB200_PIPELINE_PIECE overrides; 0 = off).
// Measured on 4 GiB of pinned host text: 43.8 GB/s upload-then-search, 51.7 GB/s pipelined
// (the PCIe rate).  tests/test_gpu_parity.py::test_pipelined_host_find_all and
// tools/micro/pipeline_probe.py compare it with the plain path.
static constexpr uint64_t kPipelinePieceDefault = 64ull << 20;

// Host haystack, pipelined: the upload is cut into pieces on a copy stream and every piece is
// searched as a byte-range shard of the (partly resident) device buffer as soon as it and
// the halo behind it have arrived, so the search hides under the PCIe transfer and the
// spans of a piece travel back while later pieces are still going up.  Pieces are taken
// left to right, so each enters the find_iter chain with its predecessor's exact exit
// state; the reverse-scan state a piece assumed at its top is checked against the exact
// one its successor computes.  Anything unusual (a wrong assumption, a match running past
// the halo) abandons the pipeline: the caller then runs the plain path on the resident text.
// Returns 0 = done, 1 = not applicable / abandoned (text is fully resident), < 0 = error.
int Regex::find_all_host_pipelined(const uint8_t* text, uint64_t n, uint8_t* d, uint64_t* d_out, uint64_t* out, uint64_t cap,
                                   uint64_t* total) {
  uint64_t piece = kPipelinePieceDefault;
  if (const char* e = getenv("RB200_PIPELINE_PIECE")) piece = (uint64_t)atoll(e) / 256 * 256;
  const uint64_t halo = 64 << 10;
  if (piece == 0 || n < 2 * piece || is_set_ || patterns_.empty()) {
    RB_CUDA(cudaMemcpyAsync(d, text, n, cudaMemcpyHostToDevice, (cudaStream_t)stream_));
    return 1;
  }
  if (int rc = side_streams()) return rc;
  cudaStream_t up = (cudaStream_t)copy_stream_, back = (cudaStream_t)back_stream_;
  const uint64_t n_pieces = (n + piece - 1) / piece;
  std::vector<cudaEvent_t> arrived(n_pieces, nullptr);
  auto cleanup = [&](int rc) {  // every exit goes through here
    cudaStreamSynchronize(up);  // the plain path needs the whole text anyway
    cudaStreamSynchronize(back);
    for (auto& e : arrived) if (e) cudaEventDestroy(e);
    return rc;
  };
#define RB_PIPE(call)                                    \
  do {                                                   \
    int rc__ = check((int)(call), #call);                \
    if (rc__) return cleanup(rc__);                      \
  } while (0)
  for (uint64_t i = 0; i < n_pieces; i++) {
    const uint64_t lo = i * piece, len = std::min(piece, n - lo);
    RB_PIPE(cudaMemcpyAsync(d + lo, text + lo, len, cudaMemcpyHostToDevice, up));
    RB_PIPE(cudaEventCreateWithFlags(&arrived[i], cudaEventDisableTiming));
    RB_PIPE(cudaEventRecord(arrived[i], up));
  }
  // scratch sized for the whole haystack up front (DeviceBuf::ensure reallocates on growth)
  if (!bitmap_.ensure(((n >> 6) + 2) * 8)) return cleanup(fail("out of device memory (bitmap)"));
  uint64_t done = 0, chain_p = 0, chain_lm = kNone;
  uint32_t prev_guess = kNoState;
  for (uint64_t i = 0; i < n_pieces; i++) {
    const uint64_t lo = i * piece, hi = std::min(n, lo + piece);
    const uint64_t n_i = std::min(n, hi + halo);  // resident prefix this piece may read
    RB_PIPE(cudaEventSynchronize(arrived[std::min(n_pieces - 1, (n_i - 1) / piece)]));
    ShardIO io;
    io.own_lo = lo;
    io.own_hi = hi;
    io.is_first = i == 0;
    io.is_last = n_i == n;
    io.chain_p = chain_p;
    io.chain_lm = chain_lm;
    uint64_t* dst = d_out && cap > done ? d_out + 2 * done : nullptr;
    const uint64_t room = cap > done ? cap - done : 0;
    const int rc = find_all_shard_device(d, n_i, &io, dst, room);
    if (rc) {
      if (io.halo_overflow) return cleanup(1);  // a match longer than the halo: do it in one piece
      return cleanup(rc);
    }
    if (i > 0 && prev_guess != io.rev_left) return cleanup(1);  // the previous piece guessed its top state wrong
    prev_guess = hi < n ? io.rev_guess : kNoState;
    if (dst) {
      const uint64_t k = std::min(room, io.n_matches);
      if (k) RB_PIPE(cudaMemcpyAsync(out + 2 * done, dst, k * 16, cudaMemcpyDeviceToHost, back));
    }
    done += io.n_matches;
    chain_p = io.exit_p;
    chain_lm = io.exit_lm;
    if (chain_p == kNone) {  // the iteration ended (a failed slice emulation): nothing further matches
      break;
    }
  }
  *total = done;
  return cleanup(0);
#undef RB_PIPE
}

int Regex::find_all_host(const uint8_t* text, uint64_t n, uint64_t start, uint64_t* out, uint64_t cap, uint64_t* total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  int rc;
  if ((rc = init_device())) return rc;
  if (use_window(n, out ? cap : 0)) return find_all_window(text, n, start, out, cap, total);  // larger than the device
  if (start == 0 && n >= (8u << 20) && out && cap) {
    if ((rc = init_device())) return rc;
    uint8_t* dd = (uint8_t*)text_.ensure(n + 64);
    uint64_t* d_out = (uint64_t*)out_.ensure(cap * 16);
    if (!dd || !d_out) return fail("out of device memory (haystack / spans)");
    DeviceDfa* warm;  // picks the stream, creates the pinned scratch
    if ((rc = ensure(kFwdAnchoredLF, &warm))) return rc;
    *total = 0;
    rc = find_all_host_pipelined(text, n, dd, d_out, out, cap, total);
    if (rc <= 0) return rc < 0 ? rc : 0;
    // not applicable or abandoned: the text is resident now, search it in one piece
    if ((rc = find_all_device(dd, n, 0, d_out, cap, total))) return rc;
    const uint64_t k = std::min(cap, *total);
    if (k) RB_CUDA(d2h(out, d_out, k * 16));
    return 0;
  }
  const uint8_t* d = upload_text(text, n, &rc);
  if (rc) return rc;
  uint64_t* d_out = nullptr;
  if (out && cap) {
    d_out = (uint64_t*)out_.ensure(cap * 16);
    if (!d_out) return fail("out of device memory (spans)");
  }
  if ((rc = find_all_device(d, n, start, d_out, cap, total))) return rc;
  const uint64_t k = std::min(cap, *total);
  if (d_out && k) RB_CUDA(d2h(out, d_out, k * 16));
  return 0;
}
// find_at on a host haystack (rure_find): the reference's cost is the distance to the next match
// (src/exec.rs:473-514), so the haystack is uploaded and searched in windows that grow from
// 64 KiB (x8 each) starting at `start`, every window as a byte-range shard entered with the
// exact iterator state of the one before, and the search stops at the first span.  A C loop
// `while (rure_find(re, h, n, pos, &m)) pos = m.end;` therefore moves each byte over PCIe
// about once per match near it instead of once per call.
int Regex::find_at_host(const uint8_t* text, uint64_t n, uint64_t start, bool* found, uint64_t* s, uint64_t* e) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *found = false;
  if (start > n) return 0;
  if (int rc = init_device()) return rc;
  if (is_set_) return fail("find requires exactly one pattern (RegexSet cannot be used with find, exec.rs:510-512)");
  uint8_t* d = (uint8_t*)text_.ensure(n + 64);
  uint64_t* d_out = (uint64_t*)out_.ensure(16);
  if (!d || !d_out) return fail("out of device memory (haystack)");
  cudaStream_t st = (cudaStream_t)stream_;
  const uint64_t buf_lo = start > 256 ? (start - 256) & ~255ull : 0;  // 256 bytes of left context for look-behind
  uint64_t resident = buf_lo;                                         // bytes [buf_lo, resident) are on the device
  uint64_t own_lo = shard_own_lo(start);
  uint64_t win = 64 << 10, halo = 64 << 10;
  uint64_t p = start, lm = kNone;
  for (;;) {
    uint64_t own_hi = std::min<uint64_t>(n, (own_lo + win + 255) & ~(uint64_t)255);
    if (n - own_hi < 4096) own_hi = n;
    const uint64_t hi = std::min(n, own_hi + halo);
    if (hi == n) own_hi = n;  // the buffer ends with the text: the last window owns everything up to it
    if (hi > resident) {
      RB_CUDA(cudaMemcpyAsync(d + resident, text + resident, hi - resident, cudaMemcpyHostToDevice, st));
      resident = hi;
    }
    ShardIO io;
    io.own_lo = own_lo - buf_lo;
    io.own_hi = own_hi - buf_lo;
    io.is_first = buf_lo == 0;
    io.is_last = hi == n;
    io.chain_p = p - buf_lo;
    io.chain_lm = lm == kNone ? kNone : lm - buf_lo;
    const int rc = find_all_shard_device(d + buf_lo, hi - buf_lo, &io, d_out, 1);
    if (rc) {
      if (!io.halo_overflow) return rc;
      if (hi == n) return rc;
      halo *= 8;  // a match longer than the halo: look further
      continue;
    }
    if (io.n_matches) {
      uint64_t h[2];
      RB_CUDA(d2h(h, d_out, 16));
      *found = true;
      *s = h[0] + buf_lo;
      *e = h[1] + buf_lo;
      return 0;
    }
    if (own_hi == n || io.exit_p == kNone) return 0;
    p = io.exit_p + buf_lo;
    lm = io.exit_lm == kNone ? kNone : io.exit_lm + buf_lo;
    own_lo = own_hi;
    win *= 8;
  }
}
// is_match / shortest_match / set matches on a host haystack: the waves of forward_reduce upload
// what they are about to read, so an early exit also ends the transfer (dfa.rs:658-667).
int Regex::shortest_match_host(const uint8_t* text, uint64_t n, uint64_t start, bool* found, uint64_t* end) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *found = false;
  if (int rc = init_device()) return rc;
  if (use_match_window(n)) return match_window(text, n, start, false, found, end, nullptr);  // larger than the device
  uint8_t* d = (uint8_t*)text_.ensure(n + 64);
  if (!d) return fail("out of device memory (haystack)");
  LazyUpload up{text, d, n, start > 256 ? (start - 256) & ~255ull : 0};
  lazy_ = &up;
  const int rc = shortest_match_device(d, n, start, found, end);
  lazy_ = nullptr;
  return rc;
}
int Regex::set_matches_host(const uint8_t* text, uint64_t n, uint64_t start, bool* any, uint64_t* masks) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *any = false;
  if (int rc = init_device()) return rc;
  if (use_match_window(n)) {  // larger than the device
    for (uint32_t w = 0; w < (patterns_.size() + 63) / 64; w++) masks[w] = 0;
    return match_window(text, n, start, true, any, nullptr, masks);
  }
  uint8_t* d = (uint8_t*)text_.ensure(n + 64);
  if (!d) return fail("out of device memory (haystack)");
  LazyUpload up{text, d, n, start > 256 ? (start - 256) & ~255ull : 0};
  lazy_ = &up;
  const int rc = set_matches_device(d, n, start, any, masks);
  lazy_ = nullptr;
  return rc;
}
int Regex::is_match_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint8_t* out_bits) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  const uint8_t* d;
  uint64_t* d_off;
  int rc = upload_batch(text, offsets, n_rec, &d, &d_off);
  if (rc) return rc;
  uint32_t* d_bits = (uint32_t*)bits_.ensure((n_rec + 31) / 32 * 4 + 4);
  if (!d_bits) return fail("out of device memory (batch)");
  if ((rc = is_match_batch_device(d, d_off, n_rec, d_bits))) return rc;
  RB_CUDA(d2h(out_bits, d_bits, (n_rec + 7) / 8));
  return 0;
}
int Regex::find_iter_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* match_offsets, uint64_t* out,
                                uint64_t cap, uint64_t* total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  const uint8_t* d;
  uint64_t* d_off;
  int rc = upload_batch(text, offsets, n_rec, &d, &d_off);
  if (rc) return rc;
  uint64_t* d_moff = (uint64_t*)bres_off_.ensure((n_rec + 1) * 8);
  if (!d_moff) return fail("out of device memory (batch)");
  if (!out) cap = 0;
  uint64_t* d_spans = cap ? (uint64_t*)out_.ensure(cap * 16) : nullptr;
  if (cap && !d_spans) return fail("out of device memory (batch spans)");
  if ((rc = find_iter_batch_device(d, d_off, n_rec, d_moff, d_spans, cap, total))) return rc;
  const uint64_t k = std::min(cap, *total);
  if (k) RB_CUDA(d2h(out, d_spans, k * 16));
  RB_CUDA(d2h(match_offsets, d_moff, (n_rec + 1) * 8));
  return 0;
}
int Regex::captures_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* slots, uint8_t* out_bits) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  const uint8_t* d;
  uint64_t* d_off;
  int rc = upload_batch(text, offsets, n_rec, &d, &d_off);
  if (rc) return rc;
  const uint64_t ns = 2 * (uint64_t)n_groups_;
  uint32_t* d_bits = (uint32_t*)bits_.ensure((n_rec + 31) / 32 * 4 + 4);
  uint64_t* d_slots = (uint64_t*)cap_slots_.ensure(std::max<uint64_t>(n_rec, 1) * ns * 8);
  if (!d_bits || !d_slots) return fail("out of device memory (batch)");
  if ((rc = captures_batch_device(d, d_off, n_rec, d_slots, d_bits))) return rc;
  RB_CUDA(d2h(out_bits, d_bits, (n_rec + 7) / 8));
  RB_CUDA(d2h(slots, d_slots, n_rec * ns * 8));
  return 0;
}
int Regex::upload_batch(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, const uint8_t** d_text, uint64_t** d_offsets) {
  int rc;
  *d_text = upload_text(text, n_rec ? offsets[n_rec] : 0, &rc);
  if (rc) return rc;
  *d_offsets = (uint64_t*)boffsets_.ensure((n_rec + 1) * 8);
  if (!*d_offsets) return fail("out of device memory (batch)");
  RB_CUDA(cudaMemcpyAsync(*d_offsets, offsets, (n_rec + 1) * 8, cudaMemcpyHostToDevice, (cudaStream_t)stream_));
  return 0;
}
int Regex::replace_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, const uint8_t* rep, uint64_t rep_len, bool expand,
                              uint64_t limit, uint64_t* out_offsets, uint8_t* out, uint64_t out_cap, uint64_t* out_len) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *out_len = 0;
  const uint8_t* d;
  uint64_t* d_off;
  if (int rc = upload_batch(text, offsets, n_rec, &d, &d_off)) return rc;
  uint64_t* d_oo = (uint64_t*)bres_off_.ensure((n_rec + 1) * 8);
  if (!d_oo) return fail("out of device memory (batch)");
  if (int rc = replace_batch_device(d, d_off, n_rec, rep, rep_len, expand, limit, d_oo, nullptr, 0, out_len)) return rc;
  const uint64_t k = out ? std::min(out_cap, *out_len) : 0;
  if (k) {
    uint8_t* d_out = (uint8_t*)bres_.ensure(*out_len);
    if (!d_out) return fail("out of device memory (replace output)");
    if (int rc = replace_emit(d_out, *out_len)) return rc;
    RB_CUDA(d2h(out, d_out, k));
  }
  RB_CUDA(d2h(out_offsets, d_oo, (n_rec + 1) * 8));
  return 0;
}
int Regex::split_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, bool has_limit, uint64_t limit, uint64_t* piece_offsets,
                            uint64_t* pieces, uint64_t cap, uint64_t* n_total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *n_total = 0;
  const uint8_t* d;
  uint64_t* d_off;
  if (int rc = upload_batch(text, offsets, n_rec, &d, &d_off)) return rc;
  if (!pieces) cap = 0;
  uint64_t* d_po = (uint64_t*)bres_off_.ensure((n_rec + 1) * 8);
  uint64_t* d_p = cap ? (uint64_t*)bres_.ensure(cap * 16) : nullptr;
  if (!d_po || (cap && !d_p)) return fail("out of device memory (batch pieces)");
  if (int rc = split_batch_device(d, d_off, n_rec, has_limit, limit, d_po, d_p, cap, n_total)) return rc;
  const uint64_t k = std::min(cap, *n_total);
  if (k) RB_CUDA(d2h(pieces, d_p, k * 16));
  RB_CUDA(d2h(piece_offsets, d_po, (n_rec + 1) * 8));
  return 0;
}
int Regex::captures_iter_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* match_offsets, uint64_t* slots,
                                    uint64_t cap, uint64_t* n_total) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  *n_total = 0;
  if (int rc = ensure_capture_program()) return rc;
  const uint8_t* d;
  uint64_t* d_off;
  if (int rc = upload_batch(text, offsets, n_rec, &d, &d_off)) return rc;
  if (!slots) cap = 0;
  const uint64_t ns = 2 * (uint64_t)n_groups_;
  uint64_t* d_mo = (uint64_t*)bres_off_.ensure((n_rec + 1) * 8);
  uint64_t* d_s = cap ? (uint64_t*)bres_.ensure(cap * ns * 8) : nullptr;
  if (!d_mo || (cap && !d_s)) return fail("out of device memory (batch captures)");
  if (int rc = captures_iter_batch_device(d, d_off, n_rec, d_mo, d_s, cap, n_total)) return rc;
  const uint64_t k = std::min(cap, *n_total);
  if (k) RB_CUDA(d2h(slots, d_s, k * ns * 8));
  RB_CUDA(d2h(match_offsets, d_mo, (n_rec + 1) * 8));
  return 0;
}
int Regex::find_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* spans, uint8_t* out_bits) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  const uint8_t* d;
  uint64_t* d_off;
  int rc = upload_batch(text, offsets, n_rec, &d, &d_off);
  if (rc) return rc;
  uint32_t* d_bits = (uint32_t*)bits_.ensure((n_rec + 31) / 32 * 4 + 4);
  uint64_t* d_spans = (uint64_t*)out_.ensure(std::max<uint64_t>(n_rec, 1) * 16);
  if (!d_bits || !d_spans) return fail("out of device memory (batch)");
  if ((rc = find_batch_device(d, d_off, n_rec, d_spans, d_bits))) return rc;
  RB_CUDA(d2h(out_bits, d_bits, (n_rec + 7) / 8));
  RB_CUDA(d2h(spans, d_spans, n_rec * 16));
  return 0;
}
int Regex::set_matches_batch_host(const uint8_t* text, const uint64_t* offsets, uint64_t n_rec, uint64_t* masks) {
  std::lock_guard<std::recursive_mutex> lock(mu_);
  const uint8_t* d;
  uint64_t* d_off;
  int rc = upload_batch(text, offsets, n_rec, &d, &d_off);
  if (rc) return rc;
  const uint32_t mw = (uint32_t)std::max<size_t>(1, (patterns_.size() + 63) / 64);
  uint64_t* d_masks = (uint64_t*)masks_.ensure(std::max<uint64_t>(n_rec, 1) * 8 * mw);
  if (!d_masks) return fail("out of device memory (batch)");
  if ((rc = set_matches_batch_device(d, d_off, n_rec, d_masks))) return rc;
  RB_CUDA(d2h(masks, d_masks, n_rec * 8 * mw));
  return 0;
}


// ------------------------------------------------------------------- streams ----
// A find_iter over text that arrives in pieces (DESIGN.md §8).  The stream's device window holds one contiguous
// buffer: at least 256 bytes of left context, the searched pieces whose spans are not final yet (the pending pieces),
// and every byte that arrived after them, which is the next piece and its halo.  Each search is one
// find_all_shard_device call on that buffer.  A piece is final, and its spans leave, once a later piece reports at
// its left edge the reverse-scan state its left neighbour assumed at its top; the pieces in between are made to
// agree first (settle), each searched again from the exact state while it is still resident.
static constexpr uint64_t kStreamPieceDefault = 64ull << 20;
static constexpr uint64_t kStreamGranule = 8ull << 20;  // most bytes per upload (and per pinned staging buffer)

// ---- the window both streams share ----
StreamWindow::~StreamWindow() {
  if (!re_) return;
  std::lock_guard<std::recursive_mutex> lock(re_->mu_);
  if (re_->copy_stream_) cudaStreamSynchronize((cudaStream_t)re_->copy_stream_);
  if (re_->stream_) cudaStreamSynchronize((cudaStream_t)re_->stream_);
  for (int k = 0; k < 2; k++) {
    if (staging_[k]) cudaFreeHost(staging_[k]);
    if (staging_ev_[k]) cudaEventDestroy((cudaEvent_t)staging_ev_[k]);
  }
  for (auto& u : uploads_) cudaEventDestroy((cudaEvent_t)u.second);
  for (void* e : free_events_) cudaEventDestroy((cudaEvent_t)e);
  if (moved_ev_) cudaEventDestroy((cudaEvent_t)moved_ev_);
}

int StreamWindow::init(Regex* re, uint64_t cap, uint64_t granule, uint64_t base, std::string* err) {
  re_ = re;
  cap_ = cap;
  granule_ = granule;
  base_ = end_ = base;
  if (re->side_streams()) {
    *err = re->error_;
    return -1;
  }
  if (!buf_.ensure(cap_ + 64)) {
    *err = "out of device memory (stream window of " + std::to_string(cap_) + " bytes)";
    return -1;
  }
  for (int k = 0; k < 2; k++) {
    cudaEvent_t ev;
    if (cudaMallocHost(&staging_[k], granule_) != cudaSuccess || cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
      *err = "out of pinned host memory (stream staging)";
      return -1;
    }
    staging_ev_[k] = ev;
  }
  cudaEvent_t ev;
  if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
    *err = "cannot create a CUDA event";
    return -1;
  }
  moved_ev_ = ev;
  return 0;
}

bool StreamWindow::pinned(const uint8_t* data, uint64_t len) {
  cudaPointerAttributes attr;
  const bool p = len && cudaPointerGetAttributes(&attr, data) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();  // a pageable pointer is not an error
  return p;
}

#define RB_WINDOW_CUDA(call)                                                                      \
  do {                                                                                            \
    const cudaError_t e__ = (call);                                                               \
    if (e__ != cudaSuccess) {                                                                     \
      *err = std::string("CUDA error in ") + #call + ": " + cudaGetErrorString(e__);              \
      return -1;                                                                                  \
    }                                                                                             \
  } while (0)

int StreamWindow::upload(const uint8_t* data, uint64_t len, bool pinned, std::string* err) {
  cudaStream_t up = (cudaStream_t)re_->copy_stream_;
  const uint8_t* src = data;
  int k = next_staging_;
  if (!pinned) {  // through pinned staging: the copy engine reads one buffer while the other is filled
    next_staging_ ^= 1;
    RB_WINDOW_CUDA(cudaEventSynchronize((cudaEvent_t)staging_ev_[k]));
    std::memcpy(staging_[k], data, len);
    src = staging_[k];
  }
  RB_WINDOW_CUDA(cudaMemcpyAsync((uint8_t*)buf_.ptr + (end_ - base_), src, len, cudaMemcpyHostToDevice, up));
  if (!pinned) RB_WINDOW_CUDA(cudaEventRecord((cudaEvent_t)staging_ev_[k], up));
  cudaEvent_t ev;
  if (!free_events_.empty()) {
    ev = (cudaEvent_t)free_events_.back();
    free_events_.pop_back();
  } else {
    RB_WINDOW_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
  end_ += len;
  uploads_.push_back({end_, ev});
  RB_WINDOW_CUDA(cudaEventRecord(ev, up));
  return 0;
}

int StreamWindow::wait_uploads(uint64_t upto, std::string* err) {
  size_t i = 0;
  while (i < uploads_.size() && uploads_[i].first < upto) i++;
  if (i == uploads_.size()) {
    if (i == 0) return 0;
    i--;
  }
  // uploads are ordered on the copy stream: waiting for the one that ends at or after upto covers those before it
  RB_WINDOW_CUDA(cudaStreamWaitEvent((cudaStream_t)re_->stream_, (cudaEvent_t)uploads_[i].second, 0));
  for (size_t j = 0; j < i; j++) free_events_.push_back(uploads_[j].second);
  uploads_.erase(uploads_.begin(), uploads_.begin() + i);
  return 0;
}

// The move runs on the engine's stream after every upload, in steps of at most the distance moved so that no copy
// overlaps itself; uploads into the freed room wait for it.
int StreamWindow::make_room(uint64_t keep_from, uint64_t want, std::string* err) {
  const uint64_t nb = std::max<uint64_t>(base_, keep_from >= 256 ? (keep_from - 256) & ~255ull : 0);
  if (cap_ - (end_ - nb) < want) {
    *err = "internal error: the stream window is full";
    return -1;
  }
  if (nb == base_) return 0;
  cudaStream_t st = (cudaStream_t)re_->stream_;
  uint8_t* w = (uint8_t*)buf_.ptr;
  const uint64_t len = end_ - nb, off = nb - base_;
  if (int rc = wait_uploads(end_, err)) return rc;
  for (uint64_t d = 0; d < len; d += off)
    RB_WINDOW_CUDA(cudaMemcpyAsync(w + d, w + off + d, std::min(off, len - d), cudaMemcpyDeviceToDevice, st));
  RB_WINDOW_CUDA(cudaEventRecord((cudaEvent_t)moved_ev_, st));
  RB_WINDOW_CUDA(cudaStreamWaitEvent((cudaStream_t)re_->copy_stream_, (cudaEvent_t)moved_ev_, 0));
  base_ = nb;
  return 0;
}
#undef RB_WINDOW_CUDA

// ---- find_iter streams ----
Stream* Stream::create(Regex* re, uint64_t piece, uint64_t hold, bool spans, uint64_t start, std::string* err) {
  std::lock_guard<std::recursive_mutex> lock(re->mu_);
  std::unique_ptr<Stream> s(new Stream(re));
  if (re->is_set_) {
    *err = "find requires exactly one pattern (RegexSet cannot be used with find, exec.rs:510-512)";
    return nullptr;
  }
  Regex::DeviceDfa* warm;  // picks the stream, creates the pinned scratch
  if (re->init_device() || re->ensure(kFwdAnchoredLF, &warm)) {
    *err = re->error_;
    return nullptr;
  }
  s->piece_ = piece ? (piece + 255) & ~255ull : kStreamPieceDefault;
  s->hold_ = hold ? (hold + 255) & ~255ull : s->piece_;
  s->halo_ = std::min<uint64_t>(64 << 10, s->hold_);
  s->granule_ = std::min(kStreamGranule, std::max<uint64_t>(256, s->piece_ / 2));
  // left context + the pending pieces + the next piece + its longest halo + the uploads in flight
  const uint64_t cap = 4096 + (kMaxPending + 1) * s->piece_ + s->hold_ + 2 * s->granule_;
  s->spans_ = spans;
  s->next_lo_ = shard_own_lo(start);
  s->chain_p_ = start;
  s->chain_lm_ = kNone;
  if (s->win_.init(re, cap, s->granule_, buf_lo(start), err)) return nullptr;
  return s.release();
}

Stream::~Stream() = default;

int Stream::fail(const std::string& msg) {
  error_ = msg;
  failed_ = true;
  return -1;
}
int Stream::cuda(int e, const char* what) {
  if (e == cudaSuccess) return 0;
  return fail(std::string("CUDA error in ") + what + ": " + cudaGetErrorString((cudaError_t)e));
}
#define RB_STREAM_CUDA(call)                            \
  do {                                                  \
    int rc__ = cuda((int)(call), #call);                \
    if (rc__) return rc__;                              \
  } while (0)

int Stream::write(const uint8_t* data, uint64_t len) {
  std::lock_guard<std::recursive_mutex> lock(re_->mu_);
  if (failed_) return -1;
  if (finished_) return fail("write after finish: the stream's text has ended");
  if (re_->init_device()) return fail(re_->error_);
  const bool pinned = StreamWindow::pinned(data, len);
  bool progressed;
  while (len && !done_) {
    const uint64_t want = std::min(len, granule_);
    if (win_.room() < want) {
      do {
        if (int rc = step(&progressed)) return rc;
      } while (progressed);
      if (win_.make_room(n_pend_ ? pend_[0].lo : next_lo_, want, &error_)) return fail(error_);
    }
    const uint64_t k = std::min(want, win_.room());
    if (win_.upload(data, k, pinned, &error_)) return fail(error_);
    data += k;
    len -= k;
  }
  do {
    if (int rc = step(&progressed)) return rc;
  } while (progressed);
  // the caller may reuse its buffer once write returns: uploads straight from it must have landed
  if (pinned) RB_STREAM_CUDA(cudaStreamSynchronize((cudaStream_t)re_->copy_stream_));
  return 0;
}

int Stream::finish() {
  std::lock_guard<std::recursive_mutex> lock(re_->mu_);
  if (failed_) return -1;
  if (finished_) return 0;
  if (re_->init_device()) return fail(re_->error_);
  finished_ = true;
  while (!done_) {
    bool progressed;
    if (int rc = step(&progressed)) return rc;
    if (!progressed) return fail("internal error: the stream cannot settle its last piece");
  }
  RB_STREAM_CUDA(cudaStreamSynchronize((cudaStream_t)re_->stream_));  // spans copied to the sink
  return 0;
}

uint64_t Stream::read(uint64_t* out, uint64_t cap) {
  const uint64_t k = std::min(cap, (queue_.size() - queue_head_) / 2);
  if (k) std::memcpy(out, queue_.data() + queue_head_, k * 16);
  queue_head_ += 2 * k;
  if (queue_head_ == queue_.size()) {
    queue_.clear();
    queue_head_ = 0;
  } else if (queue_head_ > queue_.size() / 2) {
    queue_.erase(queue_.begin(), queue_.begin() + queue_head_);
    queue_head_ = 0;
  }
  return k;
}

// One find_all_shard_device call over the window for piece p (p->lo, hi, entry_*, buf in).  Returns 1 when a match
// runs past the bytes that have arrived: the halo has grown, search again once they are there.
int Stream::search(Piece* p, uint32_t rev_entry) {
  const uint64_t base = win_.base(), end = win_.end();
  const uint64_t n_end = finished_ ? end : std::min(end, p->hi + halo_);
  if (win_.wait_uploads(n_end, &error_)) return fail(error_);
  ShardIO io;
  io.own_lo = p->lo - base;
  io.own_hi = p->hi - base;
  io.is_first = base == 0;
  io.is_last = finished_ && n_end == end;
  io.rev_entry = rev_entry;
  if (p->entry_p < base) {  // the iterator stands left of the window: enter at its first byte (sharded.py)
    io.chain_p = 0;
    io.chain_lm = kNone;
    io.chain_clamped = true;
  } else {
    io.chain_p = p->entry_p - base;
    io.chain_lm = p->entry_lm == kNone || p->entry_lm < base ? kNone : p->entry_lm - base;
  }
  p->has_spans = spans_ && !(sink_ && emitted_ >= sink_cap_);
  DeviceBuf& buf = dspan_[p->buf];
  if (p->has_spans && !buf.ensure(std::max<uint64_t>(4096, piece_ / 32) * 16)) return fail("out of device memory (stream spans)");
  for (;;) {
    uint64_t* d_out = p->has_spans ? (uint64_t*)buf.ptr : nullptr;
    const uint64_t cap = p->has_spans ? buf.cap / 16 : 0;
    if (re_->find_all_shard_device(win_.ptr(), n_end - base, &io, d_out, cap)) {
      if (io.halo_overflow && !io.is_last) {
        if (n_end - p->hi >= hold_)
          return fail("a match is longer than the stream window (" + std::to_string(hold_) + " bytes): enlarge hold");
        halo_ = std::min(hold_, (n_end - p->hi) * 8);
        return 1;
      }
      if (io.left_ctx_short)
        return fail("a look-around pattern needs text left of the stream window (" + std::to_string(p->lo - base) +
                    " bytes of left context): the iterator stands further back than the window keeps");
      return fail(re_->error_);
    }
    if (!p->has_spans || io.n_matches <= cap) break;
    // more spans than the buffer holds: grow it and search the piece again
    if (!buf.ensure(io.n_matches * 20)) return fail("out of device memory (stream spans)");
  }
  if (p->has_spans && io.n_matches) {
    cudaStream_t st = (cudaStream_t)re_->stream_;
    add_to_words<<<grid_for(2 * io.n_matches, 256, 4), 256, 0, st>>>((uint64_t*)buf.ptr, 2 * io.n_matches, base);
    g_launches++;
    RB_STREAM_CUDA(cudaGetLastError());
  }
  auto to_stream = [&](uint64_t v) { return v == kNone || v == kSpec ? v : v + base; };
  p->n = io.n_matches;
  p->rev_guess = io.rev_guess;
  p->rev_left = io.rev_left;
  p->exit_p = to_stream(io.exit_p);
  p->exit_lm = to_stream(io.exit_lm);
  return 0;
}

int Stream::step(bool* progressed) {
  *progressed = false;
  if (done_) return 0;
  Piece p;
  p.lo = next_lo_;
  p.hi = next_lo_ + piece_;
  const uint64_t end = win_.end();
  if (finished_) p.hi = std::min(p.hi, end);
  else if (end < p.hi + halo_) return 0;  // its bytes and halo have not all arrived
  const bool last = finished_ && p.hi == end;
  p.entry_p = chain_p_;
  p.entry_lm = chain_lm_;
  bool used[kMaxPending + 2] = {};
  for (int k = 0; k < n_pend_; k++) used[pend_[k].buf] = true;
  while (used[p.buf]) p.buf++;
  *progressed = true;
  if (int rc = search(&p, kNoState)) return rc < 0 ? rc : 0;
  pend_[n_pend_++] = p;
  next_lo_ = p.hi;
  chain_p_ = p.exit_p;
  chain_lm_ = p.exit_lm;
  const bool ended = last || chain_p_ == kNone;  // the text or the iteration ended (a failed slice emulation)
  // A wrong rev_left of p (p's own top guess was wrong) looks the same as a wrong guess of the piece before it, so a
  // mismatch waits for later pieces while the window holds them; a match is taken as the exact state.
  if (n_pend_ == 1 || (!ended && n_pend_ <= kMaxPending && pend_[n_pend_ - 2].rev_guess != p.rev_left)) {
    if (ended) return finish_pending();
    return 0;
  }
  if (int rc = settle()) return rc;
  if (ended) return finish_pending();
  // every piece but p is final
  for (int k = 0; k + 1 < n_pend_; k++)
    if (int rc = emit(pend_[k])) return rc;
  emitted_guess_ = pend_[n_pend_ - 2].rev_guess;
  emitted_any_ = true;
  pend_[0] = pend_[n_pend_ - 1];
  n_pend_ = 1;
  return 0;
}

int Stream::finish_pending() {
  for (int k = 0; k < n_pend_; k++)
    if (int rc = emit(pend_[k])) return rc;
  n_pend_ = 0;
  done_ = true;
  return 0;
}

// Taking the newest pending piece's rev_left as exact, make every edge between pending pieces agree: right to left,
// a piece whose top guess differs from its right neighbour's rev_left is searched again from that state (which may
// change its own rev_left), then, left to right, every piece whose entering iterator state changed is searched again.
int Stream::settle() {
  const std::string too_long = "a match is longer than the stream window (" + std::to_string(hold_) + " bytes)";
  int first = n_pend_;
  for (int k = n_pend_ - 2; k >= 0; k--) {
    if (pend_[k].rev_guess == pend_[k + 1].rev_left) continue;
    if (int rc = search(&pend_[k], pend_[k + 1].rev_left)) return rc < 0 ? rc : fail(too_long);
    first = k;
  }
  // The emitted piece before the pending ones was checked against the first pending piece's rev_left at the time;
  // spans that left cannot be taken back.  This is the only wrong guess not caught while both pieces of its edge are
  // still resident.
  if (first == 0 && emitted_any_ && pend_[0].rev_left != emitted_guess_)
    return fail("the reverse scan's state at a piece edge changed after the piece left the stream; use larger pieces");
  for (int k = std::max(first, 0) + 1; k < n_pend_; k++) {
    Piece& q = pend_[k];
    if (q.entry_p == pend_[k - 1].exit_p && q.entry_lm == pend_[k - 1].exit_lm) continue;
    q.entry_p = pend_[k - 1].exit_p;
    q.entry_lm = pend_[k - 1].exit_lm;
    if (int rc = search(&q, k + 1 < n_pend_ ? pend_[k + 1].rev_left : kNoState)) return rc < 0 ? rc : fail(too_long);
  }
  const Piece& p = pend_[n_pend_ - 1];
  chain_p_ = p.exit_p;
  chain_lm_ = p.exit_lm;
  return 0;
}

int Stream::emit(const Piece& p) {
  cudaStream_t st = (cudaStream_t)re_->stream_;
  const uint64_t* src = (const uint64_t*)dspan_[p.buf].ptr;
  if (p.has_spans && p.n && sink_) {
    const uint64_t k = std::min(p.n, sink_cap_ > emitted_ ? sink_cap_ - emitted_ : 0);
    if (k) RB_STREAM_CUDA(cudaMemcpyAsync(sink_ + 2 * emitted_, src, k * 16, cudaMemcpyDeviceToHost, st));
  } else if (p.has_spans && p.n) {
    const size_t old = queue_.size();
    queue_.resize(old + 2 * p.n);
    RB_STREAM_CUDA(cudaMemcpyAsync(queue_.data() + old, src, p.n * 16, cudaMemcpyDeviceToHost, st));
    RB_STREAM_CUDA(cudaStreamSynchronize(st));
  }
  emitted_ += p.n;
  return 0;
}
#undef RB_STREAM_CUDA

// ---- forward streams: is_match / shortest_match / RegexSet matches ----
// Each piece is one forward_step (DFA) or one cand_shortest launch (candidate starts) on the window.  Pieces after the
// first begin on multiples of 256; a DFA piece is searched once it and the 64 bytes after it have arrived (what
// forward_reduce's lazy upload brings), a candidate-start piece once look_ bytes after it have.
MatchStream* MatchStream::create(Regex* re, uint64_t piece, uint64_t hold, bool want_masks, uint64_t start, std::string* err) {
  std::lock_guard<std::recursive_mutex> lock(re->mu_);
  std::unique_ptr<MatchStream> s(new MatchStream(re));
  if (re->init_device()) {
    *err = re->error_;
    return nullptr;
  }
  s->piece_ = piece ? (piece + 255) & ~255ull : kStreamPieceDefault;
  s->hold_ = hold ? (hold + 255) & ~255ull : s->piece_;
  s->look_ = std::min<uint64_t>(64 << 10, s->hold_);
  s->want_masks_ = want_masks && re->is_set_;
  s->cand_ = re->candidate_mode();
  s->next_lo_ = start;
  s->res_.assign(re->result_words(), 0);
  s->res_[0] = kNone;
  if (!s->cand_) {
    re->forward_tabs(&s->tabs_, &s->firsts_);
    s->entries_.assign(s->tabs_.size(), kNoEntry);
    s->done_.assign(s->tabs_.size(), 0);
  }
  s->decided_ = re->patterns_.empty();  // an empty set matches nothing
  const uint64_t granule = std::min(kStreamGranule, std::max<uint64_t>(256, s->piece_ / 2));
  // left context + the piece + the bytes after it (the look-ahead, at most hold) + the uploads in flight
  const uint64_t cap = 4096 + s->piece_ + s->hold_ + 2 * granule;
  if (s->win_.init(re, cap, granule, Stream::buf_lo(start), err)) return nullptr;
  return s.release();
}

MatchStream::~MatchStream() = default;

int MatchStream::fail(const std::string& msg) {
  error_ = msg;
  failed_ = true;
  return -1;
}

bool MatchStream::found() const {
  bool any = res_[0] != kNone;
  for (size_t w = 1; w < res_.size(); w++) any = any || res_[w];
  return any;
}

int MatchStream::write(const uint8_t* data, uint64_t len) {
  std::lock_guard<std::recursive_mutex> lock(re_->mu_);
  if (failed_) return -1;
  if (finished_) return fail("write after finish: the stream's text has ended");
  if (decided_) return 0;
  if (re_->init_device()) return fail(re_->error_);
  const bool pinned = StreamWindow::pinned(data, len);
  bool progressed;
  while (len && !decided_) {
    const uint64_t want = std::min(len, win_.granule());
    if (win_.room() < want) {
      do {
        if (int rc = step(&progressed)) return rc;
      } while (progressed);
      if (decided_) break;
      if (win_.make_room(next_lo_, want, &error_)) return fail(error_);
    }
    const uint64_t k = std::min(want, win_.room());
    if (win_.upload(data, k, pinned, &error_)) return fail(error_);
    data += k;
    len -= k;
  }
  do {
    if (int rc = step(&progressed)) return rc;
  } while (progressed);
  // the caller may reuse its buffer once write returns: uploads straight from it must have landed
  if (pinned && cudaStreamSynchronize((cudaStream_t)re_->copy_stream_) != cudaSuccess) return fail("CUDA error in the stream upload");
  return 0;
}

int MatchStream::finish() {
  std::lock_guard<std::recursive_mutex> lock(re_->mu_);
  if (failed_) return -1;
  if (finished_) return 0;
  if (re_->init_device()) return fail(re_->error_);
  finished_ = true;
  while (!decided_) {
    bool progressed;
    if (int rc = step(&progressed)) return rc;
    if (!progressed) return fail("internal error: the stream cannot search its last piece");
  }
  if (cudaStreamSynchronize((cudaStream_t)re_->stream_) != cudaSuccess) return fail("CUDA error at the end of the stream");
  return 0;
}

int MatchStream::step(bool* progressed) {
  *progressed = false;
  if (decided_) return 0;
  const uint64_t end = win_.end();
  uint64_t hi = (next_lo_ & ~255ull) + piece_;
  if (finished_) hi = std::min(hi, end);
  else if (end < hi + (cand_ ? look_ : 64)) return 0;  // its bytes and the look-ahead have not all arrived
  const bool last = finished_ && hi == end;
  *progressed = true;
  bool advanced = true;
  if (int rc = cand_ ? search_cand(hi, last, &advanced) : search_dfa(hi, last)) return rc;
  if (!advanced) return 0;  // the look-ahead grew: search the piece again once its bytes are there
  next_lo_ = hi;
  re_->stats.waves = ++pieces_;
  decided_ = decided_ || last;
  return 0;
}

int MatchStream::search_dfa(uint64_t hi, bool last) {
  const uint64_t base = win_.base();
  const uint64_t n_end = finished_ ? win_.end() : hi + 64;
  if (win_.wait_uploads(n_end, &error_)) return fail(error_);
  const uint64_t n = n_end - base;
  std::vector<uint64_t> r(res_.size(), 0);
  r[0] = kNone;
  bool live;
  if (re_->forward_step(tabs_, firsts_, win_.ptr(), n, next_lo_ - base, last ? n + 1 : hi - base, want_masks_, &entries_, &done_, r.data(), &live))
    return fail(re_->error_);
  if (r[0] != kNone) res_[0] = std::min(res_[0], r[0] + base);
  for (size_t w = 1; w < r.size(); w++) res_[w] |= r[w];
  re_->stats.groups = (uint32_t)tabs_.size();
  if (want_masks_) {  // every pattern has matched, or no automaton is open (dead, or all its patterns matched)
    re_->retire_matched(firsts_, res_.data(), &done_);
    bool all = true;
    for (size_t i = 0; i < re_->patterns_.size() && all; i++) all = (res_[1 + i / 64] >> (i % 64)) & 1;
    decided_ = all || std::find(done_.begin(), done_.end(), 0) == done_.end();
  } else {  // a first match end: no later piece has an earlier one
    decided_ = !live || res_[0] != kNone;
  }
  return 0;
}

int MatchStream::search_cand(uint64_t hi, bool last, bool* advanced) {
  const uint64_t base = win_.base();
  const uint64_t n_end = finished_ ? win_.end() : hi + look_;
  if (win_.wait_uploads(n_end, &error_)) return fail(error_);
  const uint64_t n = n_end - base;
  cudaStream_t st = (cudaStream_t)re_->stream_;
  unsigned long long* best = &re_->d_scalars_->cand_best;
  uint32_t* overflow = &re_->d_scalars_->cand_overflow;
  // a bound found in an earlier piece past its end: candidates in [next_lo_, bound) may still end before it
  const uint64_t seed = res_[0] == kNone ? kNone : res_[0] - base;
  if (cudaMemcpyAsync(best, &seed, 8, cudaMemcpyHostToDevice, st) != cudaSuccess || cudaMemsetAsync(overflow, 0, 4, st) != cudaSuccess)
    return fail("CUDA error in the stream's candidate search");
  if (re_->cand_shortest_range(win_.ptr(), n, next_lo_ - base, last ? n + 1 : hi - base, !finished_, best, overflow)) return fail(re_->error_);
  uint64_t b = kNone;
  uint32_t o = 0;
  if (re_->d2h(&b, best, 8) || re_->d2h(&o, overflow, 4)) return fail("CUDA error in the stream's candidate search");
  if (o && b == kNone) {
    // a run reached the end of the window undecided: read further past the piece, up to hold bytes
    if (look_ >= hold_) return fail("a match is longer than the stream window (" + std::to_string(hold_) + " bytes): enlarge hold");
    look_ = std::min(hold_, look_ * 8);
    *advanced = false;
    return 0;
  }
  if (b != kNone) res_[0] = b + base;
  decided_ = res_[0] != kNone && res_[0] <= hi;  // every later candidate, and so its end, lies at or after hi
  return 0;
}

bool Regex::use_match_window(uint64_t n) {
  if (tuning.host_window) return n > tuning.host_window;
  if (text_.ensure(n + 64)) return false;  // the buffer the resident path takes anyway
  cudaGetLastError();  // the failed allocation is not an error of a later call
  return true;
}

// shortest_match_host / set_matches_host through a MatchStream: the text goes up piece by piece and stops at the
// piece that decides the answer.
int Regex::match_window(const uint8_t* text, uint64_t n, uint64_t start, bool want_masks, bool* found, uint64_t* end, uint64_t* masks) {
  *found = false;
  if (start > n) return 0;
  const uint64_t w = tuning.host_window;
  const uint64_t piece = w ? std::max<uint64_t>(256, w / 8 / 256 * 256) : kStreamPieceDefault;
  std::string err;
  std::unique_ptr<MatchStream> s(MatchStream::create(this, piece, w ? piece : 4 * kStreamPieceDefault, want_masks, start, &err));
  if (!s) return fail(err);
  const uint64_t lo = Stream::buf_lo(start);
  if (s->write(text + lo, n - lo) || s->finish()) return fail(s->error());
  *found = s->found();
  if (*found && end) *end = s->end();
  if (masks)
    for (uint32_t i = 0; i < (patterns_.size() + 63) / 64; i++) masks[i] = s->mask()[i];
  return 0;
}

bool Regex::use_window(uint64_t n, uint64_t cap) {
  if (tuning.host_window) return n > tuning.host_window;
  // The buffers the whole-haystack paths take anyway: the haystack, its start bitmap and the spans.
  if (text_.ensure(n + 64) && bitmap_.ensure(((n >> 6) + 2) * 8) && (cap == 0 || out_.ensure(cap * 16))) return false;
  cudaGetLastError();  // the failed allocation is not an error of a later call
  return true;
}

int Regex::find_all_window(const uint8_t* text, uint64_t n, uint64_t start, uint64_t* out, uint64_t cap, uint64_t* total) {
  *total = 0;
  if (start > n) return 0;  // re_trait.rs:198-200
  const uint64_t w = tuning.host_window;
  const uint64_t piece = w ? std::max<uint64_t>(256, w / 8 / 256 * 256) : kStreamPieceDefault;
  std::string err;
  std::unique_ptr<Stream> s(Stream::create(this, piece, w ? piece : 4 * kStreamPieceDefault, out && cap, start, &err));
  if (!s) return fail(err);
  s->sink(out, cap);
  const uint64_t lo = Stream::buf_lo(start);
  if (s->write(text + lo, n - lo) || s->finish()) return fail(s->error());
  *total = s->count();
  return 0;
}

}  // namespace rbgpu
