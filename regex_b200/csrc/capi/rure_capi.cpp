// extern "C" surface declared in include/rure.h and include/rure_b200.h.
// Thin: argument checks, object lifetime, and calls into rbgpu::Regex.
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../../include/rure_b200.h"
#include "../gpu/engine.h"

using rbgpu::Regex;

struct rure_options {
  size_t size_limit = 10u << 20;
  size_t dfa_size_limit = 2u << 20;
};
struct rure_error {
  std::string msg = "no error";
};
// rure.h:27-34: a compiled regex may be used from several threads at once.  The engine keeps its device
// scratch (bitmap, staging, counters, stream) per object, so a scalar call that finds the object busy takes a
// clone compiled from the same source; the clones stay with the handle.  Bulk, device and shard entry points
// run on the primary engine and serialise.
struct EnginePool {
  Regex* re = nullptr;  // primary
  std::vector<std::string> pats;
  rbgpu::CompileOptions opts;
  std::mutex mu;
  std::vector<Regex*> clones;
  ~EnginePool() {
    for (Regex* c : clones) delete c;
    delete re;
  }
};
struct rure : EnginePool {};
struct rure_set : EnginePool {};
struct Lease {
  Regex* r;
  explicit Lease(EnginePool* h) {
    if (h->re->try_acquire()) { r = h->re; return; }
    std::lock_guard<std::mutex> g(h->mu);
    for (Regex* c : h->clones)
      if (c->try_acquire()) { r = c; return; }
    rb::Error err;
    Regex* c = h->re->clone(&err);  // a grouped set compiles its planned groups, not the failed product automaton
    if (!c) {  // cannot happen for a source that compiled once; wait for the primary then
      h->re->acquire();
      r = h->re;
      return;
    }
    c->tuning = h->re->tuning;
    c->acquire();
    h->clones.push_back(c);
    r = c;
  }
  ~Lease() { r->release(); }
  Regex* operator->() const { return r; }
};
struct rure_captures {
  size_t n_groups = 1;
  bool has = false;
  std::vector<uint64_t> slots;  // 2 per group, ~0 = the group did not take part
};
struct rure_iter {
  rure* re;
  size_t last_end = 0;
  bool has_last_match = false;
  size_t last_match = 0;
  // all spans of the haystack seen on the first call (see rure.h)
  const uint8_t* hay = nullptr;
  size_t len = 0;
  bool cached = false;
  std::vector<rure_match> spans;
  size_t next = 0;
  std::vector<uint64_t> slots;  // capture slots of every cached span (filled by the first rure_iter_next_captures)
  bool have_slots = false;
};
struct rure_iter_capture_names {
  std::vector<std::string> names;  // one per group, "" = unnamed
  size_t next = 0;
  std::vector<char*> handed_out;
};

static thread_local std::string g_last_error;

static bool ok(Regex* re, int rc) {
  if (rc == 0) return true;
  g_last_error = re->last_error();
  return false;
}
// The scalar reference API cannot report runtime failures (Rust panics abort,
// regex-capi/src/macros.rs:11-27); a search that cannot run on the GPU does the same.
[[noreturn]] static void die(const char* where) {
  std::fprintf(stderr, "regex_b200: %s failed: %s\n", where, g_last_error.c_str());
  std::abort();
}

template <typename Handle>
static Handle* compile_common(const std::vector<std::string>& pats, uint32_t flags, rure_options* options,
                              rure_error* error, bool only_utf8, bool as_set) {
  rbgpu::CompileOptions o;
  o.flags = flags;
  o.only_utf8 = only_utf8;
  o.as_set = as_set;
  if (options) { o.size_limit = options->size_limit; o.dfa_size_limit = options->dfa_size_limit; }
  rb::Error err;
  Regex* re = Regex::compile(pats, o, &err);
  if (!re) {
    if (error) error->msg = err.msg;
    g_last_error = err.msg;
    return nullptr;
  }
  Handle* h = new Handle();
  h->re = re;
  h->pats = pats;
  h->opts = o;
  return h;
}

extern "C" {

rure* rure_compile(const uint8_t* pattern, size_t length, uint32_t flags, rure_options* options, rure_error* error) {
  return compile_common<rure>({std::string((const char*)pattern, length)}, flags, options, error, false, false);
}
rure* rure_b200_compile_str(const uint8_t* pattern, size_t length, uint32_t flags, rure_options* options, rure_error* error) {
  return compile_common<rure>({std::string((const char*)pattern, length)}, flags, options, error, true, false);
}
rure* rure_compile_must(const char* pattern) {
  rure_error err;
  rure* r = rure_compile((const uint8_t*)pattern, std::strlen(pattern), RURE_DEFAULT_FLAGS, nullptr, &err);
  if (!r) {
    std::fprintf(stderr, "%s\naborting from rure_compile_must\n", err.msg.c_str());
    std::abort();
  }
  return r;
}
void rure_free(rure* re) { delete re; }

bool rure_is_match(rure* re, const uint8_t* haystack, size_t length, size_t start) {
  bool found = false;
  uint64_t end = 0;
  Lease l(re);
  if (!ok(l.r, l->shortest_match_host(haystack, length, start, &found, &end))) die("rure_is_match");
  return found;
}
bool rure_shortest_match(rure* re, const uint8_t* haystack, size_t length, size_t start, size_t* end) {
  bool found = false;
  uint64_t e = 0;
  Lease l(re);
  if (!ok(l.r, l->shortest_match_host(haystack, length, start, &found, &e))) die("rure_shortest_match");
  if (found && end) *end = e;
  return found;
}
bool rure_find(rure* re, const uint8_t* haystack, size_t length, size_t start, rure_match* match) {
  bool found = false;
  uint64_t s = 0, e = 0;
  Lease l(re);
  if (!ok(l.r, l->find_at_host(haystack, length, start, &found, &s, &e))) die("rure_find");
  if (found && match) { match->start = s; match->end = e; }
  return found;
}
bool rure_find_captures(rure* re, const uint8_t* haystack, size_t length, size_t start, rure_captures* captures) {
  bool found = false;
  std::vector<uint64_t> slots(2 * (size_t)re->re->n_groups(), ~0ull);
  Lease l(re);
  if (!ok(l.r, l->captures_at_host(haystack, length, start, &found, slots.data()))) die("rure_find_captures");
  if (captures) {
    captures->has = found;
    captures->slots = found ? slots : std::vector<uint64_t>(slots.size(), ~0ull);
  }
  return found;
}
int32_t rure_capture_name_index(rure* re, const char* name) {
  if (!name) return -1;
  for (const auto& g : re->re->group_names())
    if (g.first == name) return g.second;
  return -1;
}
rure_iter_capture_names* rure_iter_capture_names_new(rure* re) {
  auto* it = new rure_iter_capture_names();
  it->names.assign((size_t)re->re->n_groups(), "");
  for (const auto& g : re->re->group_names()) it->names[(size_t)g.second] = g.first;
  return it;
}
void rure_iter_capture_names_free(rure_iter_capture_names* it) {
  if (!it) return;
  for (char* p : it->handed_out) std::free(p);
  delete it;
}
bool rure_iter_capture_names_next(rure_iter_capture_names* it, char** name) {
  if (!name || it->next >= it->names.size()) return false;
  char* p = strdup(it->names[it->next++].c_str());  // owned by the iterator, like the reference's CString::into_raw list
  it->handed_out.push_back(p);
  *name = p;
  return true;
}

rure_iter* rure_iter_new(rure* re) {
  rure_iter* it = new rure_iter();
  it->re = re;
  return it;
}
void rure_iter_free(rure_iter* it) { delete it; }
bool rure_iter_next(rure_iter* it, const uint8_t* haystack, size_t length, rure_match* match) {
  if (!it->cached || it->hay != haystack || it->len != length) {
    // Continue the chain from last_end on this haystack: find_iter restarted at
    // last_end is exactly the remaining sequence (re_trait.rs:197-220).
    it->hay = haystack;
    it->len = length;
    it->spans.clear();
    it->next = 0;
    it->cached = true;
    if (it->last_end <= length) {
      uint64_t total = 0;
      size_t cap = 1 << 12;
      for (;;) {
        it->spans.resize(cap);
        if (!ok(it->re->re, it->re->re->find_all_host(haystack, length, it->last_end, (uint64_t*)it->spans.data(), cap, &total)))
          die("rure_iter_next");
        if (total <= cap) break;
        cap = total;
      }
      it->spans.resize(total);
      // The empty-match skip rule depends on the previous match of this iterator.
      if (it->has_last_match && !it->spans.empty() && it->spans[0].start == it->spans[0].end &&
          it->spans[0].end == it->last_match)
        it->next = 1;
    }
  }
  if (it->next >= it->spans.size()) {
    it->last_end = length + 1;
    return false;
  }
  const rure_match m = it->spans[it->next++];
  it->last_end = (m.start == m.end) ? m.end + 1 : m.end;
  it->has_last_match = true;
  it->last_match = m.end;
  if (match) *match = m;
  return true;
}
bool rure_iter_next_captures(rure_iter* it, const uint8_t* haystack, size_t length, rure_captures* captures) {
  rure_match m;
  const size_t before = it->next;
  const bool found = rure_iter_next(it, haystack, length, &m);
  if (!captures) return found;
  const size_t ns = 2 * (size_t)it->re->re->n_groups();
  captures->has = found;
  captures->slots.assign(ns, ~0ull);
  if (!found) return false;
  if (!it->have_slots) {  // the groups of every cached span in one pass
    uint64_t total = 0;
    it->slots.assign(std::max<size_t>(it->spans.size(), 1) * ns, ~0ull);
    if (!ok(it->re->re, it->re->re->captures_all_host(haystack, length, it->slots.data(), it->spans.size(), &total))) die("rure_iter_next_captures");
    it->have_slots = true;
  }
  // the cached spans are find_iter from the iterator's position at caching time; the capture pass saw the same list
  size_t idx = it->next - 1;
  (void)before;
  if (it->slots.size() >= (idx + 1) * ns && it->slots[idx * ns] == m.start && it->slots[idx * ns + 1] == m.end) {
    std::copy(it->slots.begin() + idx * ns, it->slots.begin() + (idx + 1) * ns, captures->slots.begin());
  } else {  // an iterator that started mid-haystack: ask for this match alone
    bool f2 = false;
    if (!ok(it->re->re, it->re->re->captures_at_host(haystack, length, m.start, &f2, captures->slots.data()))) die("rure_iter_next_captures");
  }
  return true;
}

rure_captures* rure_captures_new(rure* re) {
  auto* c = new rure_captures();
  c->n_groups = (size_t)re->re->n_groups();
  c->slots.assign(2 * c->n_groups, ~0ull);
  return c;
}
void rure_captures_free(rure_captures* c) { delete c; }
bool rure_captures_at(rure_captures* c, size_t i, rure_match* match) {
  if (!c->has || i >= c->n_groups || c->slots[2 * i] == ~0ull || c->slots[2 * i + 1] == ~0ull) return false;
  if (match) { match->start = c->slots[2 * i]; match->end = c->slots[2 * i + 1]; }
  return true;
}
size_t rure_captures_len(rure_captures* c) { return c->n_groups; }

// every match with all its groups: slots[i][2 * n_groups], SIZE_MAX where a group did not take part
bool rure_b200_captures_all(rure* re, const uint8_t* haystack, size_t length, size_t* slots, size_t cap, size_t* n_matches, size_t* n_groups) {
  uint64_t m = 0;
  if (n_groups) *n_groups = (size_t)re->re->n_groups();
  const bool r = ok(re->re, re->re->captures_all_host(haystack, length, (uint64_t*)slots, slots ? cap : 0, &m));
  if (n_matches) *n_matches = m;
  return r;
}
bool rure_b200_captures(rure* re, const uint8_t* haystack, size_t length, size_t start, bool* found, size_t* slots) {
  Lease l(re);
  return ok(l.r, l->captures_at_host(haystack, length, start, found, (uint64_t*)slots));
}
size_t rure_b200_captures_len(rure* re) { return (size_t)re->re->n_groups(); }

rure_options* rure_options_new(void) { return new rure_options(); }
void rure_options_free(rure_options* o) { delete o; }
void rure_options_size_limit(rure_options* o, size_t limit) { o->size_limit = limit; }
void rure_options_dfa_size_limit(rure_options* o, size_t limit) { o->dfa_size_limit = limit; }

rure_set* rure_compile_set(const uint8_t** patterns, const size_t* lengths, size_t count, uint32_t flags,
                           rure_options* options, rure_error* error) {
  std::vector<std::string> pats;
  for (size_t i = 0; i < count; i++) pats.emplace_back((const char*)patterns[i], lengths[i]);
  return compile_common<rure_set>(pats, flags, options, error, false, true);
}
rure_set* rure_b200_compile_set_str(const uint8_t** patterns, const size_t* lengths, size_t count, uint32_t flags,
                                    rure_options* options, rure_error* error) {
  std::vector<std::string> pats;
  for (size_t i = 0; i < count; i++) pats.emplace_back((const char*)patterns[i], lengths[i]);
  return compile_common<rure_set>(pats, flags, options, error, true, true);
}
void rure_set_free(rure_set* s) { delete s; }
bool rure_set_is_match(rure_set* s, const uint8_t* haystack, size_t length, size_t start) {
  bool found = false;
  uint64_t end = 0;
  Lease l(s);
  if (!ok(l.r, l->shortest_match_host(haystack, length, start, &found, &end))) die("rure_set_is_match");
  return found;
}
bool rure_set_matches(rure_set* s, const uint8_t* haystack, size_t length, size_t start, bool* matches) {
  const size_t n = s->re->n_patterns();
  for (size_t i = 0; i < n; i++) matches[i] = false;
  std::vector<uint64_t> masks(std::max<size_t>(1, (n + 63) / 64), 0);
  bool any = false;
  Lease l(s);
  if (!ok(l.r, l->set_matches_host(haystack, length, start, &any, masks.data()))) die("rure_set_matches");
  for (size_t i = 0; i < n; i++) matches[i] = (masks[i / 64] >> (i % 64)) & 1;
  return any;
}
size_t rure_set_len(rure_set* s) { return s->re->n_patterns(); }

rure_error* rure_error_new(void) { return new rure_error(); }
void rure_error_free(rure_error* e) { delete e; }
const char* rure_error_message(rure_error* e) { return e->msg.c_str(); }

// ---------------------------------------- scalar searches that report failures --
// The reference's scalar entry points cannot fail at run time, so rure_is_match & co abort when
// the GPU search cannot run (no device, out of memory).  Hosts that prefer an error code use these.
bool rure_b200_is_match(rure* re, const uint8_t* haystack, size_t length, size_t start, bool* matched) {
  uint64_t end = 0;
  Lease l(re);
  return ok(l.r, l->shortest_match_host(haystack, length, start, matched, &end));
}
bool rure_b200_shortest_match(rure* re, const uint8_t* haystack, size_t length, size_t start, bool* found, size_t* end) {
  uint64_t e = 0;
  Lease l(re);
  const bool r = ok(l.r, l->shortest_match_host(haystack, length, start, found, &e));
  if (r && *found && end) *end = e;
  return r;
}
bool rure_b200_find(rure* re, const uint8_t* haystack, size_t length, size_t start, bool* found, rure_match* match) {
  uint64_t s = 0, e = 0;
  Lease l(re);
  const bool r = ok(l.r, l->find_at_host(haystack, length, start, found, &s, &e));
  if (r && *found && match) { match->start = s; match->end = e; }
  return r;
}
bool rure_b200_set_is_match(rure_set* set, const uint8_t* haystack, size_t length, size_t start, bool* matched) {
  uint64_t end = 0;
  Lease l(set);
  return ok(l.r, l->shortest_match_host(haystack, length, start, matched, &end));
}

// ------------------------------------------------------------ bulk extension --
bool rure_b200_find_all(rure* re, const uint8_t* haystack, size_t length, rure_match* out, size_t cap, size_t* n_total) {
  uint64_t total = 0;
  bool r = ok(re->re, re->re->find_all_host(haystack, length, 0, (uint64_t*)out, out ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_count_all(rure* re, const uint8_t* haystack, size_t length, size_t* n_total) {
  return rure_b200_find_all(re, haystack, length, nullptr, 0, n_total);
}
bool rure_b200_set_matches_mask(rure_set* s, const uint8_t* haystack, size_t length, size_t start, uint64_t* mask_words) {
  bool any;
  return ok(s->re, s->re->set_matches_host(haystack, length, start, &any, mask_words));
}
bool rure_b200_is_match_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, uint8_t* out_bits) {
  return ok(re->re, re->re->is_match_batch_host(haystack, offsets, n, out_bits));
}
bool rure_b200_find_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, rure_match* out, uint8_t* found_bits) {
  return ok(re->re, re->re->find_batch_host(haystack, offsets, n, (uint64_t*)out, found_bits));
}
bool rure_b200_set_matches_batch(rure_set* s, const uint8_t* haystack, const uint64_t* offsets, size_t n, uint64_t* out_masks) {
  return ok(s->re, s->re->set_matches_batch_host(haystack, offsets, n, out_masks));
}
bool rure_b200_find_iter_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, uint64_t* match_offsets, rure_match* out,
                               size_t cap, size_t* n_total) {
  uint64_t total = 0;
  const bool r = ok(re->re, re->re->find_iter_batch_host(haystack, offsets, n, match_offsets, (uint64_t*)out, out ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_find_iter_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, uint64_t* d_match_offsets,
                                      rure_match* d_out, size_t cap, size_t* n_total) {
  uint64_t total = 0;
  const bool r = ok(re->re, re->re->find_iter_batch_device(d_haystack, d_offsets, n, d_match_offsets, (uint64_t*)d_out, d_out ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_captures_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, size_t* slots, uint8_t* found_bits) {
  return ok(re->re, re->re->captures_batch_host(haystack, offsets, n, (uint64_t*)slots, found_bits));
}
bool rure_b200_captures_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, size_t* d_slots,
                                     uint32_t* d_found_bits) {
  return ok(re->re, re->re->captures_batch_device(d_haystack, d_offsets, n, (uint64_t*)d_slots, d_found_bits));
}
bool rure_b200_replace_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, const uint8_t* rep, size_t rep_len, int expand,
                             size_t limit, uint64_t* out_offsets, uint8_t* out, size_t out_cap, size_t* out_len) {
  uint64_t ol = 0;
  const bool r = ok(re->re, re->re->replace_batch_host(haystack, offsets, n, rep, rep_len, expand != 0, limit, out_offsets, out, out ? out_cap : 0, &ol));
  if (out_len) *out_len = ol;
  return r;
}
bool rure_b200_replace_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, const uint8_t* rep, size_t rep_len,
                                    int expand, size_t limit, uint64_t* d_out_offsets, uint8_t* d_out, size_t out_cap, size_t* out_len) {
  uint64_t ol = 0;
  const bool r = ok(re->re, re->re->replace_batch_device(d_haystack, d_offsets, n, rep, rep_len, expand != 0, limit, d_out_offsets, d_out,
                                                         d_out ? out_cap : 0, &ol));
  if (out_len) *out_len = ol;
  return r;
}
bool rure_b200_split_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, int has_limit, size_t limit, uint64_t* piece_offsets,
                           rure_match* out, size_t cap, size_t* n_total) {
  uint64_t total = 0;
  const bool r = ok(re->re, re->re->split_batch_host(haystack, offsets, n, has_limit != 0, limit, piece_offsets, (uint64_t*)out, out ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_split_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, int has_limit, size_t limit,
                                  uint64_t* d_piece_offsets, rure_match* d_out, size_t cap, size_t* n_total) {
  uint64_t total = 0;
  const bool r = ok(re->re, re->re->split_batch_device(d_haystack, d_offsets, n, has_limit != 0, limit, d_piece_offsets, (uint64_t*)d_out,
                                                       d_out ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_captures_iter_batch(rure* re, const uint8_t* haystack, const uint64_t* offsets, size_t n, uint64_t* match_offsets, size_t* slots,
                                   size_t cap, size_t* n_total) {
  uint64_t total = 0;
  const bool r = ok(re->re, re->re->captures_iter_batch_host(haystack, offsets, n, match_offsets, (uint64_t*)slots, slots ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_captures_iter_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, uint64_t* d_match_offsets,
                                          size_t* d_slots, size_t cap, size_t* n_total) {
  uint64_t total = 0;
  const bool r = ok(re->re, re->re->captures_iter_batch_device(d_haystack, d_offsets, n, d_match_offsets, (uint64_t*)d_slots, d_slots ? cap : 0,
                                                               &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_find_all_device(rure* re, const uint8_t* d_haystack, size_t length, size_t start, rure_match* d_out, size_t cap, size_t* n_total) {
  uint64_t total = 0;
  bool r = ok(re->re, re->re->find_all_device(d_haystack, length, start, (uint64_t*)d_out, d_out ? cap : 0, &total));
  if (n_total) *n_total = total;
  return r;
}
bool rure_b200_shortest_match_device(rure* re, const uint8_t* d_haystack, size_t length, size_t start, bool* found, size_t* end) {
  uint64_t e = 0;
  bool f = false;
  bool r = ok(re->re, re->re->shortest_match_device(d_haystack, length, start, &f, &e));
  if (found) *found = f;
  if (f && end) *end = e;
  return r;
}
bool rure_b200_set_matches_device(rure_set* s, const uint8_t* d_haystack, size_t length, size_t start, uint64_t* mask_words) {
  bool any;
  return ok(s->re, s->re->set_matches_device(d_haystack, length, start, &any, mask_words));
}
bool rure_b200_is_match_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, uint32_t* d_out_bits) {
  return ok(re->re, re->re->is_match_batch_device(d_haystack, d_offsets, n, d_out_bits));
}
bool rure_b200_find_batch_device(rure* re, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, rure_match* d_out, uint32_t* d_found_bits) {
  return ok(re->re, re->re->find_batch_device(d_haystack, d_offsets, n, (uint64_t*)d_out, d_found_bits));
}
bool rure_b200_set_matches_batch_device(rure_set* s, const uint8_t* d_haystack, const uint64_t* d_offsets, size_t n, uint64_t* d_out_masks) {
  return ok(s->re, s->re->set_matches_batch_device(d_haystack, d_offsets, n, d_out_masks));
}

bool rure_b200_find_all_shard_device(rure* re, const uint8_t* d_buffer, size_t n_buffer, rure_b200_shard* io, rure_match* d_out, size_t cap) {
  rbgpu::ShardIO s;
  s.own_lo = io->own_lo; s.own_hi = io->own_hi;
  s.is_first = io->is_first != 0; s.is_last = io->is_last != 0;
  s.rev_entry = io->rev_entry; s.reuse_scan = io->reuse_scan != 0;
  s.chain_p = io->chain_p; s.chain_lm = io->chain_lm;
  s.chain_clamped = io->chain_clamped != 0;
  bool r = ok(re->re, re->re->find_all_shard_device(d_buffer, n_buffer, &s, (uint64_t*)d_out, d_out ? cap : 0));
  io->rev_guess = s.rev_guess; io->rev_left = s.rev_left;
  io->exit_p = s.exit_p; io->exit_lm = s.exit_lm;
  io->n_matches = s.n_matches; io->halo_overflow = (s.halo_overflow ? 1u : 0u) | (s.left_ctx_short ? 2u : 0u);
  return r;
}

static bool forward_shard(Regex* r, const uint8_t* d_buffer, size_t n_buffer, rure_b200_fwd_shard* io, bool want_masks) {
  bool found = false;
  uint64_t first = ~0ull;
  uint32_t used = io->entry_state, exit_state = io->entry_state;
  for (auto& m : io->masks) m = 0;
  bool r_ok = ok(r, r->forward_shard_device(d_buffer, n_buffer, io->own_lo, io->own_hi, io->is_first != 0, io->is_last != 0, io->entry_state,
                                           want_masks, &found, &first, io->masks, &used, &exit_state));
  io->found = found ? 1 : 0;
  io->first_end = first;
  io->entry_used = used;
  io->exit_state = exit_state;
  return r_ok;
}
bool rure_b200_shortest_match_shard_device(rure* re, const uint8_t* d_buffer, size_t n_buffer, rure_b200_fwd_shard* io) {
  return forward_shard(re->re, d_buffer, n_buffer, io, false);
}
bool rure_b200_set_matches_shard_device(rure_set* set, const uint8_t* d_buffer, size_t n_buffer, rure_b200_fwd_shard* io) {
  return forward_shard(set->re, d_buffer, n_buffer, io, true);
}

// ---- replace_all / replacen / split / splitn (src/re_bytes.rs:316-360, 476-535) ----
bool rure_b200_replace(rure* re, const uint8_t* haystack, size_t length, const uint8_t* rep, size_t rep_len, int expand, size_t limit,
                       uint8_t* out, size_t out_cap, size_t* out_len) {
  uint64_t ol = 0;
  const bool r = ok(re->re, re->re->replace_host(haystack, length, rep, rep_len, expand != 0, limit, out, out ? out_cap : 0, &ol));
  if (out_len) *out_len = ol;
  return r;
}
bool rure_b200_replace_device(rure* re, const uint8_t* d_haystack, size_t length, const uint8_t* rep, size_t rep_len, int expand,
                              size_t limit, uint8_t* d_out, size_t out_cap, size_t* out_len) {
  uint64_t ol = 0;
  const bool r = ok(re->re, re->re->replace_device(d_haystack, length, rep, rep_len, expand != 0, limit, d_out, d_out ? out_cap : 0, &ol));
  if (out_len) *out_len = ol;
  return r;
}
bool rure_b200_split(rure* re, const uint8_t* haystack, size_t length, int has_limit, size_t limit, rure_match* out, size_t cap,
                     size_t* n_pieces) {
  uint64_t np = 0;
  const bool r = ok(re->re, re->re->split_host(haystack, length, has_limit != 0, limit, (uint64_t*)out, out ? cap : 0, &np));
  if (n_pieces) *n_pieces = np;
  return r;
}
bool rure_b200_split_device(rure* re, const uint8_t* d_haystack, size_t length, int has_limit, size_t limit, rure_match* d_out, size_t cap,
                            size_t* n_pieces) {
  uint64_t np = 0;
  const bool r = ok(re->re, re->re->split_device(d_haystack, length, has_limit != 0, limit, (uint64_t*)d_out, d_out ? cap : 0, &np));
  if (n_pieces) *n_pieces = np;
  return r;
}

const char* rure_b200_last_error(void) { return g_last_error.c_str(); }
uint64_t rure_b200_kernel_launches(void) { return rbgpu::kernel_launches(); }
void rure_b200_last_stats(rure* re, double* out8) {
  double* out7 = out8;
  out8[7] = re->re->stats.fused ? 1.0 : 0.0;
  const rbgpu::Stats& s = re->re->stats;
  out7[0] = s.scan_ms; out7[1] = s.walk_ms; out7[2] = s.total_ms;
  out7[3] = (double)s.scan_redo_rounds; out7[4] = (double)s.scan_redo_segments;
  out7[5] = (double)s.stitch_rounds; out7[6] = (double)s.stitch_dirty_chunks;
}
static void stats_ex(Regex* r, double* out, size_t n) {
  const rbgpu::Stats& s = r->stats;
  const double v[14] = {s.scan_ms, s.walk_ms, s.total_ms, (double)s.scan_redo_rounds, (double)s.scan_redo_segments,
                        (double)s.stitch_rounds, (double)s.stitch_dirty_chunks, s.fused ? 1.0 : 0.0,
                        (double)s.sequential_passes, (double)s.map_passes, (double)s.waves, (double)s.path,
                        (double)s.long_runs, (double)s.groups};
  for (size_t i = 0; i < n && i < 14; i++) out[i] = v[i];
}
void rure_b200_last_stats_ex(rure* re, double* out, size_t n) { stats_ex(re->re, out, n); }
void rure_b200_set_last_stats_ex(rure_set* set, double* out, size_t n) { stats_ex(set->re, out, n); }
static bool set_option(Regex* r, const char* name, uint64_t value) {
  rbgpu::Tuning& t = r->tuning;
  const std::string k(name ? name : "");
  if (k == "wave0") t.wave0 = value;
  else if (k == "narrow_sets") t.narrow_sets = value != 0;
  else if (k == "batch_refill") t.batch_refill = (int)value;
  else if (k == "max_stitch_rounds") t.max_stitch_rounds = (uint32_t)value;
  else if (k == "max_redo_rounds") t.max_redo_rounds = (uint32_t)value;
  else if (k == "prefilter") t.prefilter = (int)value;
  else if (k == "candidate_starts") t.candidate_starts = value != 0;
  else { g_last_error = "unknown option: " + k; return false; }
  return true;
}
bool rure_b200_set_option(rure* re, const char* name, uint64_t value) { return set_option(re->re, name, value); }
bool rure_b200_set_set_option(rure_set* set, const char* name, uint64_t value) {
  if (name && std::string(name) == "set_group_patterns") {
    if (value > 0xFFFFFFFFull) { g_last_error = "set_group_patterns: value out of range"; return false; }
    std::lock_guard<std::mutex> g(set->mu);
    if (!ok(set->re, set->re->set_group_patterns((uint32_t)value))) return false;
    for (Regex* c : set->clones) {  // clones take the new plan the next time they are needed
      c->acquire();
      c->release();
      delete c;
    }
    set->clones.clear();
    return true;
  }
  return set_option(set->re, name, value);
}
size_t rure_b200_set_groups(rure_set* set, size_t* first_pattern, size_t cap) {
  const std::vector<uint32_t> f = set->re->group_firsts();
  for (size_t i = 0; i < f.size() && i < cap && first_pattern; i++) first_pattern[i] = f[i];
  return f.size();
}
void rure_b200_set_tuning(rure* re, uint32_t seg, uint32_t chunk, uint32_t warm, uint32_t block, uint32_t blocks_per_sm) {
  rbgpu::Tuning& t = re->re->tuning;
  if (seg) t.seg = (seg + 63) / 64 * 64;
  if (chunk) t.chunk = (chunk + 255) / 256 * 256;
  t.warm = warm;
  if (block) t.block = (block + 31) / 32 * 32;
  if (blocks_per_sm) t.blocks_per_sm = blocks_per_sm;
}
void rure_b200_set_stream(rure* re, void* cuda_stream) { re->re->set_stream(cuda_stream); }
void rure_b200_set_set_stream(rure_set* set, void* cuda_stream) { set->re->set_stream(cuda_stream); }
void rure_b200_force_generic(rure* re, int yes) { re->re->tuning.force_generic = yes != 0; }
void rure_b200_set_fuse(rure* re, int yes) { re->re->tuning.fuse = yes != 0; }
void rure_b200_set_tensor_tma(rure* re, int yes) { re->re->tuning.tensor_tma = yes != 0; }
bool rure_b200_dfa_export(rure* re, int kind, uint32_t* info6, uint16_t* trans, uint8_t* classes, uint16_t* start, uint64_t* masks) {
  if (kind < 0 || kind >= rbgpu::kNumDfaKinds) { g_last_error = "bad dfa kind"; return false; }
  rb::Error err;
  const rb::Dfa* d = re->re->host_dfa((rbgpu::DfaKind)kind, &err);
  if (!d) { g_last_error = err.msg; return false; }
  if (info6) {
    info6[0] = d->n_states; info6[1] = d->n_classes; info6[2] = d->match_lo; info6[3] = d->mask_words;
    info6[4] = d->uniform_start; info6[5] = (uint32_t)d->raw_states;
  }
  if (trans) std::memcpy(trans, d->trans.data(), d->trans.size() * 2);
  if (classes) std::memcpy(classes, d->classes, 256);
  if (start) std::memcpy(start, d->start, sizeof d->start);
  if (masks) std::memcpy(masks, d->masks.data(), d->masks.size() * 8);
  return true;
}
void rure_b200_pattern_info(rure* re, uint64_t* info4) {
  info4[0] = re->re->min_len; info4[1] = re->re->max_len;
  info4[2] = re->re->can_match_empty; info4[3] = re->re->has_looks;
}

}  // extern "C"
