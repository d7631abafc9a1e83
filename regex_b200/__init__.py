"""regex_b200 -- B200-native search backend with the reference crate's search surface.

Python host mirror of the reference API for the search hot path (names and argument
meaning follow the Rust crate: `Regex` src/re_unicode.rs, `bytes::Regex` src/re_bytes.rs,
`RegexSet` src/re_set.rs, `RegexBuilder` src/re_builder.rs).  Every search call goes
through the C ABI in include/rure.h / include/rure_b200.h into hand-written sm_100a
kernels; there is no CPU matching path -- loading fails loudly when the CUDA
library has not been built, and searching fails loudly without a GPU.
"""
import ctypes
import os
import sys
from ctypes import POINTER, byref, c_bool, c_char_p, c_double, c_int, c_size_t, c_uint8, c_uint16, c_uint32, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "librure_b200.so")

FLAG_CASEI, FLAG_MULTI, FLAG_DOTNL, FLAG_SWAP_GREED, FLAG_SPACE, FLAG_UNICODE = 1, 2, 4, 8, 16, 32

DFA_FWD_ANCHORED_LF, DFA_REV_UNANCHORED_ALL, DFA_FWD_UNANCHORED_ALL, DFA_REV_ANCHORED_LONGEST, DFA_FWD_UNANCHORED_LF = range(5)


_STAT_KEYS = ["scan_ms", "walk_ms", "total_ms", "scan_redo_rounds", "scan_redo_segments", "stitch_rounds", "stitch_dirty_chunks",
              "fused", "sequential_passes", "map_passes", "waves", "path", "long_runs"]
_SET_STAT_KEYS = _STAT_KEYS + ["groups"]


class Error(Exception):
    """Compile error (syntax, size limit, unsupported construct) or GPU runtime error."""


class _Match(ctypes.Structure):
    _fields_ = [("start", c_size_t), ("end", c_size_t)]


class _Shard(ctypes.Structure):  # include/rure_b200.h: rure_b200_shard
    _fields_ = [("own_lo", c_uint64), ("own_hi", c_uint64), ("is_first", ctypes.c_int32), ("is_last", ctypes.c_int32),
                ("rev_entry", c_uint32), ("reuse_scan", c_uint32), ("chain_p", c_uint64), ("chain_lm", c_uint64),
                ("rev_guess", c_uint32), ("rev_left", c_uint32), ("exit_p", c_uint64), ("exit_lm", c_uint64),
                ("n_matches", c_uint64), ("halo_overflow", c_uint32), ("chain_clamped", c_uint32)]


class _FwdShard(ctypes.Structure):  # include/rure_b200.h: rure_b200_fwd_shard
    _fields_ = [("own_lo", c_uint64), ("own_hi", c_uint64), ("is_first", ctypes.c_int32), ("is_last", ctypes.c_int32),
                ("entry_state", c_uint32), ("entry_used", c_uint32), ("exit_state", c_uint32), ("found", c_uint32),
                ("first_end", c_uint64), ("masks", c_uint64 * 4)]


def _forward_shard(fn, handle, d_buffer, io):
    sh = _FwdShard(own_lo=io["own_lo"], own_hi=io["own_hi"], is_first=int(io["is_first"]), is_last=int(io["is_last"]),
                   entry_state=io["entry_state"])
    if not fn(handle, d_buffer.data_ptr(), d_buffer.numel(), byref(sh)):
        raise Error(_last_error())
    return dict(entry_used=sh.entry_used, exit_state=sh.exit_state, found=bool(sh.found), first_end=sh.first_end, masks=list(sh.masks))


def _load():
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"{_LIB_PATH} is missing: build it with `python regex_b200/build.py` "
            "(nvcc, sm_100a).  regex_b200 has no CPU fallback.")
    L = ctypes.CDLL(_LIB_PATH)
    vp, sz, u8p = c_void_p, c_size_t, c_void_p
    sig = {
        "rure_compile": (vp, [c_char_p, sz, c_uint32, vp, vp]),
        "rure_b200_compile_str": (vp, [c_char_p, sz, c_uint32, vp, vp]),
        "rure_compile_must": (vp, [c_char_p]),
        "rure_free": (None, [vp]),
        "rure_is_match": (c_bool, [vp, u8p, sz, sz]),
        "rure_find": (c_bool, [vp, u8p, sz, sz, POINTER(_Match)]),
        "rure_shortest_match": (c_bool, [vp, u8p, sz, sz, POINTER(sz)]),
        "rure_iter_new": (vp, [vp]),
        "rure_iter_free": (None, [vp]),
        "rure_iter_next": (c_bool, [vp, u8p, sz, POINTER(_Match)]),
        "rure_options_new": (vp, []),
        "rure_options_free": (None, [vp]),
        "rure_options_size_limit": (None, [vp, sz]),
        "rure_options_dfa_size_limit": (None, [vp, sz]),
        "rure_compile_set": (vp, [POINTER(c_char_p), POINTER(sz), sz, c_uint32, vp, vp]),
        "rure_b200_compile_set_str": (vp, [POINTER(c_char_p), POINTER(sz), sz, c_uint32, vp, vp]),
        "rure_set_free": (None, [vp]),
        "rure_set_is_match": (c_bool, [vp, u8p, sz, sz]),
        "rure_set_matches": (c_bool, [vp, u8p, sz, sz, POINTER(c_bool)]),
        "rure_set_len": (sz, [vp]),
        "rure_error_new": (vp, []),
        "rure_error_free": (None, [vp]),
        "rure_error_message": (c_char_p, [vp]),
        "rure_b200_is_match": (c_bool, [vp, u8p, sz, sz, POINTER(c_bool)]),
        "rure_b200_shortest_match": (c_bool, [vp, u8p, sz, sz, POINTER(c_bool), POINTER(sz)]),
        "rure_b200_find": (c_bool, [vp, u8p, sz, sz, POINTER(c_bool), POINTER(_Match)]),
        "rure_b200_set_is_match": (c_bool, [vp, u8p, sz, sz, POINTER(c_bool)]),
        "rure_b200_replace": (c_bool, [vp, u8p, sz, c_char_p, sz, c_int, sz, vp, sz, POINTER(sz)]),
        "rure_b200_replace_device": (c_bool, [vp, vp, sz, c_char_p, sz, c_int, sz, vp, sz, POINTER(sz)]),
        "rure_b200_split": (c_bool, [vp, u8p, sz, c_int, sz, vp, sz, POINTER(sz)]),
        "rure_b200_split_device": (c_bool, [vp, vp, sz, c_int, sz, vp, sz, POINTER(sz)]),
        "rure_b200_captures_len": (sz, [vp]),
        "rure_b200_captures": (c_bool, [vp, u8p, sz, sz, POINTER(c_bool), vp]),
        "rure_b200_captures_all": (c_bool, [vp, u8p, sz, vp, sz, POINTER(sz), POINTER(sz)]),
        "rure_capture_name_index": (ctypes.c_int32, [vp, c_char_p]),
        "rure_b200_find_all": (c_bool, [vp, u8p, sz, vp, sz, POINTER(sz)]),
        "rure_b200_count_all": (c_bool, [vp, u8p, sz, POINTER(sz)]),
        "rure_b200_set_matches_mask": (c_bool, [vp, u8p, sz, sz, POINTER(c_uint64)]),
        "rure_b200_is_match_batch": (c_bool, [vp, u8p, vp, sz, vp]),
        "rure_b200_find_batch": (c_bool, [vp, u8p, vp, sz, vp, vp]),
        "rure_b200_set_matches_batch": (c_bool, [vp, u8p, vp, sz, vp]),
        "rure_b200_find_iter_batch": (c_bool, [vp, u8p, vp, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_captures_batch": (c_bool, [vp, u8p, vp, sz, vp, vp]),
        "rure_b200_replace_batch": (c_bool, [vp, u8p, vp, sz, c_char_p, sz, c_int, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_split_batch": (c_bool, [vp, u8p, vp, sz, c_int, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_captures_iter_batch": (c_bool, [vp, u8p, vp, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_find_all_device": (c_bool, [vp, vp, sz, sz, vp, sz, POINTER(sz)]),
        "rure_b200_find_all_shard_device": (c_bool, [vp, vp, sz, POINTER(_Shard), vp, sz]),
        "rure_b200_shortest_match_device": (c_bool, [vp, vp, sz, sz, POINTER(c_bool), POINTER(sz)]),
        "rure_b200_shortest_match_shard_device": (c_bool, [vp, vp, sz, POINTER(_FwdShard)]),
        "rure_b200_set_matches_shard_device": (c_bool, [vp, vp, sz, POINTER(_FwdShard)]),
        "rure_b200_set_matches_device": (c_bool, [vp, vp, sz, sz, POINTER(c_uint64)]),
        "rure_b200_is_match_batch_device": (c_bool, [vp, vp, vp, sz, vp]),
        "rure_b200_find_batch_device": (c_bool, [vp, vp, vp, sz, vp, vp]),
        "rure_b200_set_matches_batch_device": (c_bool, [vp, vp, vp, sz, vp]),
        "rure_b200_find_iter_batch_device": (c_bool, [vp, vp, vp, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_captures_batch_device": (c_bool, [vp, vp, vp, sz, vp, vp]),
        "rure_b200_replace_batch_device": (c_bool, [vp, vp, vp, sz, c_char_p, sz, c_int, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_split_batch_device": (c_bool, [vp, vp, vp, sz, c_int, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_captures_iter_batch_device": (c_bool, [vp, vp, vp, sz, vp, vp, sz, POINTER(sz)]),
        "rure_b200_last_error": (c_char_p, []),
        "rure_b200_kernel_launches": (c_uint64, []),
        "rure_b200_last_stats": (None, [vp, POINTER(c_double)]),
        "rure_b200_last_stats_ex": (None, [vp, POINTER(c_double), sz]),
        "rure_b200_set_last_stats_ex": (None, [vp, POINTER(c_double), sz]),
        "rure_b200_set_option": (c_bool, [vp, c_char_p, c_uint64]),
        "rure_b200_set_set_option": (c_bool, [vp, c_char_p, c_uint64]),
        "rure_b200_set_groups": (sz, [vp, POINTER(sz), sz]),
        "rure_b200_set_tuning": (None, [vp, c_uint32, c_uint32, c_uint32, c_uint32, c_uint32]),
        "rure_b200_force_generic": (None, [vp, c_int]),
        "rure_b200_set_stream": (None, [vp, vp]),
        "rure_b200_set_set_stream": (None, [vp, vp]),
        "rure_b200_set_fuse": (None, [vp, c_int]),
        "rure_b200_set_tensor_tma": (None, [vp, c_int]),
        "rure_b200_dfa_export": (c_bool, [vp, c_int, POINTER(c_uint32), vp, vp, vp, vp]),
        "rure_b200_pattern_info": (None, [vp, POINTER(c_uint64)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    return L


def _building():
    """`python -m regex_b200.build` imports this package before the library exists."""
    return "regex_b200.build" in getattr(sys, "orig_argv", [])


_lib = None if (_building() and not os.path.exists(_LIB_PATH)) else _load()


def lib():
    return _lib


def exported_symbols():
    """Names every header in include/ declares (used by the no-GPU load test)."""
    return sorted(n for n in dir(_lib) if n.startswith("rure"))


def kernel_launches():
    return int(_lib.rure_b200_kernel_launches())


def _last_error():
    return (_lib.rure_b200_last_error() or b"").decode("utf-8", "replace")


def _buf(data):
    """bytes-like -> (pointer, length, keepalive)."""
    if isinstance(data, str):
        data = data.encode("utf-8")
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data, dtype=np.uint8) if data.dtype != np.uint8 or not data.flags.c_contiguous else data
        return a.ctypes.data, a.size, a
    if isinstance(data, (bytes, bytearray, memoryview)):
        b = bytes(data) if not isinstance(data, bytes) else data
        return ctypes.cast(c_char_p(b), c_void_p).value or 0, len(b), b
    if hasattr(data, "data_ptr"):  # pinned / CPU torch tensor
        return data.data_ptr(), data.numel() * data.element_size(), data
    raise TypeError(f"unsupported haystack type {type(data)!r}")


class RegexBuilder:
    """Options mirror src/re_builder.rs:14-40."""

    def __init__(self, pattern):
        self.pattern = pattern
        self._flags = FLAG_UNICODE
        self._size_limit = 10 << 20
        self._dfa_size_limit = 2 << 20

    def _flag(self, bit, yes):
        self._flags = (self._flags | bit) if yes else (self._flags & ~bit)
        return self

    def case_insensitive(self, yes): return self._flag(FLAG_CASEI, yes)
    def multi_line(self, yes): return self._flag(FLAG_MULTI, yes)
    def dot_matches_new_line(self, yes): return self._flag(FLAG_DOTNL, yes)
    def swap_greed(self, yes): return self._flag(FLAG_SWAP_GREED, yes)
    def ignore_whitespace(self, yes): return self._flag(FLAG_SPACE, yes)
    def unicode(self, yes): return self._flag(FLAG_UNICODE, yes)

    def size_limit(self, n):
        self._size_limit = n
        return self

    def dfa_size_limit(self, n):
        self._dfa_size_limit = n
        return self

    def build(self):
        return Regex(self.pattern, flags=self._flags, size_limit=self._size_limit, dfa_size_limit=self._dfa_size_limit)

    def build_bytes(self):
        return BytesRegex(self.pattern, flags=self._flags, size_limit=self._size_limit, dfa_size_limit=self._dfa_size_limit)


class _Compiled:
    _only_utf8 = False

    def __init__(self, pattern, flags=FLAG_UNICODE, size_limit=10 << 20, dfa_size_limit=2 << 20):
        self.pattern = pattern
        pat = pattern.encode("utf-8") if isinstance(pattern, str) else bytes(pattern)
        opts = _lib.rure_options_new()
        _lib.rure_options_size_limit(opts, size_limit)
        _lib.rure_options_dfa_size_limit(opts, dfa_size_limit)
        err = _lib.rure_error_new()
        fn = _lib.rure_b200_compile_str if self._only_utf8 else _lib.rure_compile
        self._h = fn(pat, len(pat), flags, opts, err)
        msg = _lib.rure_error_message(err).decode("utf-8", "replace")
        _lib.rure_error_free(err)
        _lib.rure_options_free(opts)
        if not self._h:
            raise Error(msg)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and _lib is not None:  # module globals are gone at interpreter shutdown
            _lib.rure_free(h)
            self._h = None

    # ---- scalar API (re_bytes.rs:141-623 / re_unicode.rs) -------------------
    def is_match(self, text):
        return self.is_match_at(text, 0)

    def is_match_at(self, text, start):
        p, n, keep = _buf(text)
        out = c_bool()
        if not _lib.rure_b200_is_match(self._h, p, n, start, byref(out)):  # the error-reporting twin of rure_is_match
            raise Error(_last_error())
        return bool(out.value)

    def shortest_match(self, text):
        return self.shortest_match_at(text, 0)

    def shortest_match_at(self, text, start):
        p, n, keep = _buf(text)
        end, found = c_size_t(), c_bool()
        if not _lib.rure_b200_shortest_match(self._h, p, n, start, byref(found), byref(end)):
            raise Error(_last_error())
        return end.value if found.value else None

    def find(self, text):
        return self.find_at(text, 0)

    def find_at(self, text, start):
        p, n, keep = _buf(text)
        m, found = _Match(), c_bool()
        if not _lib.rure_b200_find(self._h, p, n, start, byref(found), byref(m)):
            raise Error(_last_error())
        return (m.start, m.end) if found.value else None

    def find_iter(self, text):
        """All non-overlapping leftmost-first matches as a list of (start, end)."""
        return [tuple(r) for r in self.find_all(text).tolist()]

    # ---- bulk API (include/rure_b200.h) --------------------------------------
    def find_all(self, text, cap=None):
        """(n, 2) uint64 array of spans; equals collecting find_iter."""
        p, n, keep = _buf(text)
        total = c_size_t()
        cap = 4096 if cap is None else cap
        while True:
            out = np.empty((max(cap, 1), 2), dtype=np.uint64)
            if not _lib.rure_b200_find_all(self._h, p, n, out.ctypes.data, cap, byref(total)):
                raise Error(_last_error())
            if total.value <= cap:
                return out[: total.value]
            cap = total.value

    # ---- capture groups (re_bytes.rs:226-262 captures / captures_iter) ----------------
    def captures_len(self):
        """Number of capture groups, group 0 included (`Regex::captures_len`)."""
        return int(_lib.rure_b200_captures_len(self._h))

    def capture_name_index(self, name):
        i = int(_lib.rure_capture_name_index(self._h, name.encode("utf-8")))
        return None if i < 0 else i

    def captures_at(self, text, start=0):
        """`Regex::captures`: [(start, end) or None for every group], or None without a match."""
        p, n, keep = _buf(text)
        g = self.captures_len()
        slots = np.empty(2 * g, dtype=np.uint64)
        found = c_bool()
        if not _lib.rure_b200_captures(self._h, p, n, start, byref(found), slots.ctypes.data):
            raise Error(_last_error())
        if not found.value:
            return None
        none = np.uint64(0xFFFFFFFFFFFFFFFF)
        return [None if slots[2 * i] == none else (int(slots[2 * i]), int(slots[2 * i + 1])) for i in range(g)]

    def captures(self, text):
        return self.captures_at(text, 0)

    def captures_all(self, text):
        """`Regex::captures_iter` in one pass: uint64 [n_matches, n_groups, 2], 2**64-1 where a group did not take part."""
        p, n, keep = _buf(text)
        m, g = c_size_t(), c_size_t()
        if not _lib.rure_b200_captures_all(self._h, p, n, None, 0, byref(m), byref(g)):
            raise Error(_last_error())
        out = np.empty((max(m.value, 1), g.value, 2), dtype=np.uint64)
        if m.value and not _lib.rure_b200_captures_all(self._h, p, n, out.ctypes.data, m.value, byref(m), byref(g)):
            raise Error(_last_error())
        return out[:m.value]

    def captures_iter(self, text):
        none = 0xFFFFFFFFFFFFFFFF
        return [[None if int(a) == none else (int(a), int(b)) for a, b in row] for row in self.captures_all(text)]

    # ---- replace / split (re_bytes.rs:316-360, 440-535) -----------------------------
    def replacen(self, text, limit, rep, expand=True):
        """`Regex::replacen`: at most `limit` matches replaced (0 = all).  rep: bytes/str; with
        expand (the default for a plain replacement string, as in the reference) `$0`, `${0}`,
        `$$` are expanded; expand=False is `NoExpand(rep)`."""
        p, n, keep = _buf(text)
        r = rep.encode("utf-8") if isinstance(rep, str) else bytes(rep)
        ol = c_size_t()
        if not _lib.rure_b200_replace(self._h, p, n, r, len(r), int(expand), limit, None, 0, byref(ol)):
            raise Error(_last_error())
        out = np.empty(max(ol.value, 1), dtype=np.uint8)
        if not _lib.rure_b200_replace(self._h, p, n, r, len(r), int(expand), limit, out.ctypes.data, ol.value, byref(ol)):
            raise Error(_last_error())
        return out[:ol.value].tobytes()

    def replace(self, text, rep, expand=True):
        return self.replacen(text, 1, rep, expand)

    def replace_all(self, text, rep, expand=True):
        return self.replacen(text, 0, rep, expand)

    def replace_all_device(self, d_text, rep, d_out=None, expand=True, limit=0):
        """Device-resident replace_all: returns the output length; writes into d_out (uint8 CUDA tensor) when given."""
        r = rep.encode("utf-8") if isinstance(rep, str) else bytes(rep)
        ol = c_size_t()
        ptr, cap = (0, 0) if d_out is None else (d_out.data_ptr(), d_out.numel())
        if not _lib.rure_b200_replace_device(self._h, d_text.data_ptr(), d_text.numel(), r, len(r), int(expand), limit, ptr, cap, byref(ol)):
            raise Error(_last_error())
        return ol.value

    def _split(self, text, has_limit, limit):
        p, n, keep = _buf(text)
        k = c_size_t()
        if not _lib.rure_b200_split(self._h, p, n, has_limit, limit, None, 0, byref(k)):
            raise Error(_last_error())
        out = np.empty((max(k.value, 1), 2), dtype=np.uint64)
        if not _lib.rure_b200_split(self._h, p, n, has_limit, limit, out.ctypes.data, k.value, byref(k)):
            raise Error(_last_error())
        data = bytes(keep) if not isinstance(keep, bytes) else keep
        return [data[int(a):int(b)] for a, b in out[:k.value]]

    def split(self, text):
        """`Regex::split`: the pieces of text between the matches."""
        return self._split(text, 0, 0)

    def splitn(self, text, limit):
        """`Regex::splitn`: at most `limit` pieces, the last one being the rest of the text."""
        return self._split(text, 1, limit)

    def count_all(self, text):
        p, n, keep = _buf(text)
        total = c_size_t()
        if not _lib.rure_b200_count_all(self._h, p, n, byref(total)):
            raise Error(_last_error())
        return total.value

    def is_match_batch(self, text, offsets):
        """bool array, one per record text[offsets[i]:offsets[i+1]]."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        bits = np.zeros((n_rec + 7) // 8 + 8, dtype=np.uint8)
        if not _lib.rure_b200_is_match_batch(self._h, p, off.ctypes.data, n_rec, bits.ctypes.data):
            raise Error(_last_error())
        return np.unpackbits(bits, bitorder="little")[:n_rec].astype(bool)

    def find_batch(self, text, offsets):
        """(found bool[n], spans uint64[n,2]) with record-relative offsets."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        bits = np.zeros((n_rec + 7) // 8 + 8, dtype=np.uint8)
        spans = np.zeros((max(n_rec, 1), 2), dtype=np.uint64)
        if not _lib.rure_b200_find_batch(self._h, p, off.ctypes.data, n_rec, spans.ctypes.data, bits.ctypes.data):
            raise Error(_last_error())
        return np.unpackbits(bits, bitorder="little")[:n_rec].astype(bool), spans[:n_rec]

    def find_iter_batch(self, text, offsets, cap=None):
        """find_iter over every record: (match_offsets uint64[n+1], spans uint64[m, 2]); the spans of record i
        are spans[match_offsets[i]:match_offsets[i+1]], relative to the record."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        moff = np.zeros(n_rec + 1, dtype=np.uint64)
        total = c_size_t()
        cap = max(4096, 2 * n_rec) if cap is None else cap
        while True:
            out = np.empty((max(cap, 1), 2), dtype=np.uint64)
            if not _lib.rure_b200_find_iter_batch(self._h, p, off.ctypes.data, n_rec, moff.ctypes.data, out.ctypes.data, cap, byref(total)):
                raise Error(_last_error())
            if total.value <= cap:
                return moff, out[: total.value]
            cap = total.value

    def count_batch(self, text, offsets):
        """uint64[n]: the number of find_iter matches of every record (no spans are stored)."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        moff = np.zeros(n_rec + 1, dtype=np.uint64)
        total = c_size_t()
        if not _lib.rure_b200_find_iter_batch(self._h, p, off.ctypes.data, n_rec, moff.ctypes.data, None, 0, byref(total)):
            raise Error(_last_error())
        return np.diff(moff)

    def captures_batch(self, text, offsets):
        """`Regex::captures` on every record: (found bool[n], slots uint64[n, captures_len, 2]), record-relative,
        2**64-1 where a group did not take part."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        g = self.captures_len()
        bits = np.zeros((n_rec + 7) // 8 + 8, dtype=np.uint8)
        slots = np.empty((max(n_rec, 1), g, 2), dtype=np.uint64)
        if not _lib.rure_b200_captures_batch(self._h, p, off.ctypes.data, n_rec, slots.ctypes.data, bits.ctypes.data):
            raise Error(_last_error())
        return np.unpackbits(bits, bitorder="little")[:n_rec].astype(bool), slots[:n_rec]

    def replacen_batch(self, text, offsets, limit, rep, expand=True):
        """`replacen` on every record: (out_offsets uint64[n+1], out uint8[...]); record i's result is
        out[out_offsets[i]:out_offsets[i+1]].  limit applies to every record (0 = all matches); rep / expand as
        replacen."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        r = rep.encode("utf-8") if isinstance(rep, str) else bytes(rep)
        ooff = np.zeros(n_rec + 1, dtype=np.uint64)
        ol = c_size_t()
        cap = n + 4096
        while True:
            out = np.empty(max(cap, 1), dtype=np.uint8)
            if not _lib.rure_b200_replace_batch(self._h, p, off.ctypes.data, n_rec, r, len(r), int(expand), limit, ooff.ctypes.data,
                                                out.ctypes.data, cap, byref(ol)):
                raise Error(_last_error())
            if ol.value <= cap:
                return ooff, out[: ol.value]
            cap = ol.value

    def replace_batch(self, text, offsets, rep, expand=True):
        return self.replacen_batch(text, offsets, 1, rep, expand)

    def replace_all_batch(self, text, offsets, rep, expand=True):
        return self.replacen_batch(text, offsets, 0, rep, expand)

    def _split_batch(self, text, offsets, has_limit, limit):
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        poff = np.zeros(n_rec + 1, dtype=np.uint64)
        total = c_size_t()
        cap = max(4096, 2 * n_rec)
        while True:
            out = np.empty((max(cap, 1), 2), dtype=np.uint64)
            if not _lib.rure_b200_split_batch(self._h, p, off.ctypes.data, n_rec, has_limit, limit, poff.ctypes.data, out.ctypes.data, cap,
                                              byref(total)):
                raise Error(_last_error())
            if total.value <= cap:
                return poff, out[: total.value]
            cap = total.value

    def split_batch(self, text, offsets):
        """`split` on every record: (piece_offsets uint64[n+1], pieces uint64[m, 2]); the pieces of record i are
        pieces[piece_offsets[i]:piece_offsets[i+1]], relative to the record."""
        return self._split_batch(text, offsets, 0, 0)

    def splitn_batch(self, text, offsets, limit):
        """`splitn` on every record, as split_batch: at most `limit` pieces per record, the last one being the rest."""
        return self._split_batch(text, offsets, 1, limit)

    def captures_iter_batch(self, text, offsets):
        """`captures_iter` on every record: (match_offsets uint64[n+1], slots uint64[m, captures_len, 2]); the
        matches of record i are slots[match_offsets[i]:match_offsets[i+1]], relative to the record, 2**64-1 where
        a group did not take part."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        g = self.captures_len()
        moff = np.zeros(n_rec + 1, dtype=np.uint64)
        total = c_size_t()
        cap = max(4096, 2 * n_rec)
        while True:
            out = np.empty((max(cap, 1), g, 2), dtype=np.uint64)
            if not _lib.rure_b200_captures_iter_batch(self._h, p, off.ctypes.data, n_rec, moff.ctypes.data, out.ctypes.data, cap, byref(total)):
                raise Error(_last_error())
            if total.value <= cap:
                return moff, out[: total.value]
            cap = total.value

    # ---- device-resident (torch CUDA tensors) --------------------------------
    def find_all_device(self, d_text, d_out=None, start=0):
        """d_text: uint8 CUDA tensor; d_out: optional (cap, 2) int64/uint64 CUDA tensor.
        Returns the total number of matches (spans beyond cap are counted, not stored)."""
        total = c_size_t()
        cap = 0 if d_out is None else d_out.shape[0]
        ptr = 0 if d_out is None else d_out.data_ptr()
        if not _lib.rure_b200_find_all_device(self._h, d_text.data_ptr(), d_text.numel(), start, ptr, cap, byref(total)):
            raise Error(_last_error())
        return total.value

    def find_all_shard_device(self, d_buffer, io, d_out=None):
        """One shard of a sharded haystack (see regex_b200/sharded.py).  `io` carries the
        in-fields of rure_b200_shard; returns its out-fields as a dict."""
        sh = _Shard(own_lo=io["own_lo"], own_hi=io["own_hi"], is_first=int(io["is_first"]), is_last=int(io["is_last"]),
                    rev_entry=io["rev_entry"], reuse_scan=int(io["reuse_scan"]), chain_p=io["chain_p"], chain_lm=io["chain_lm"],
                    chain_clamped=int(io.get("chain_clamped", False)))
        cap = 0 if d_out is None else d_out.shape[0]
        ptr = 0 if d_out is None else d_out.data_ptr()
        if not _lib.rure_b200_find_all_shard_device(self._h, d_buffer.data_ptr(), d_buffer.numel(), byref(sh), ptr, cap):
            raise Error(_last_error())
        return dict(rev_guess=sh.rev_guess, rev_left=sh.rev_left, exit_p=sh.exit_p, exit_lm=sh.exit_lm, n_matches=sh.n_matches)

    def forward_shard_device(self, d_buffer, io):
        """is_match / shortest_match over one shard (regex_b200/sharded.py: forward_sharded)."""
        return _forward_shard(_lib.rure_b200_shortest_match_shard_device, self._h, d_buffer, io)

    def shortest_match_device(self, d_text, start=0):
        found, end = c_bool(), c_size_t()
        if not _lib.rure_b200_shortest_match_device(self._h, d_text.data_ptr(), d_text.numel(), start, byref(found), byref(end)):
            raise Error(_last_error())
        return end.value if found.value else None

    def is_match_batch_device(self, d_text, d_offsets, d_bits):
        """d_bits: int32 CUDA tensor of (n_records + 31) // 32 ballot words."""
        n_rec = d_offsets.numel() - 1
        if not _lib.rure_b200_is_match_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, d_bits.data_ptr()):
            raise Error(_last_error())

    def find_batch_device(self, d_text, d_offsets, d_spans, d_bits):
        n_rec = d_offsets.numel() - 1
        if not _lib.rure_b200_find_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, d_spans.data_ptr(), d_bits.data_ptr()):
            raise Error(_last_error())

    def find_iter_batch_device(self, d_text, d_offsets, d_match_offsets, d_out=None):
        """find_iter over every record on the device.  d_match_offsets: (n_records + 1) int64/uint64 CUDA
        tensor, always filled; d_out: optional (cap, 2) tensor for the spans (beyond cap they are counted,
        not stored).  Returns the total number of matches."""
        n_rec = d_offsets.numel() - 1
        total = c_size_t()
        cap = 0 if d_out is None else d_out.shape[0]
        ptr = 0 if d_out is None else d_out.data_ptr()
        if not _lib.rure_b200_find_iter_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, d_match_offsets.data_ptr(),
                                                     ptr, cap, byref(total)):
            raise Error(_last_error())
        return total.value

    def captures_batch_device(self, d_text, d_offsets, d_slots, d_bits):
        """d_slots: n_records * 2 * captures_len() int64/uint64 CUDA tensor; d_bits: int32 ballot words."""
        n_rec = d_offsets.numel() - 1
        if not _lib.rure_b200_captures_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, d_slots.data_ptr(), d_bits.data_ptr()):
            raise Error(_last_error())

    def replacen_batch_device(self, d_text, d_offsets, limit, rep, d_out_offsets, d_out=None, expand=True):
        """replacen_batch on the device.  d_out_offsets: (n_records + 1) int64/uint64 CUDA tensor, always filled;
        d_out: optional uint8 CUDA tensor (beyond its size the output is counted, not stored).  Returns the total
        output length."""
        n_rec = d_offsets.numel() - 1
        r = rep.encode("utf-8") if isinstance(rep, str) else bytes(rep)
        ol = c_size_t()
        ptr, cap = (0, 0) if d_out is None else (d_out.data_ptr(), d_out.numel())
        if not _lib.rure_b200_replace_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, r, len(r), int(expand), limit,
                                                   d_out_offsets.data_ptr(), ptr, cap, byref(ol)):
            raise Error(_last_error())
        return ol.value

    def split_batch_device(self, d_text, d_offsets, d_piece_offsets, d_out=None, limit=None):
        """split_batch (splitn_batch when limit is given) on the device.  d_piece_offsets: (n_records + 1) CUDA
        tensor, always filled; d_out: optional (cap, 2) tensor for the pieces.  Returns the total number of pieces."""
        n_rec = d_offsets.numel() - 1
        total = c_size_t()
        cap = 0 if d_out is None else d_out.shape[0]
        ptr = 0 if d_out is None else d_out.data_ptr()
        if not _lib.rure_b200_split_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, int(limit is not None), limit or 0,
                                                 d_piece_offsets.data_ptr(), ptr, cap, byref(total)):
            raise Error(_last_error())
        return total.value

    def captures_iter_batch_device(self, d_text, d_offsets, d_match_offsets, d_slots=None):
        """captures_iter_batch on the device.  d_match_offsets: (n_records + 1) CUDA tensor, always filled; d_slots:
        optional (cap, captures_len(), 2) tensor.  Returns the total number of matches."""
        n_rec = d_offsets.numel() - 1
        total = c_size_t()
        cap = 0 if d_slots is None else d_slots.shape[0]
        ptr = 0 if d_slots is None else d_slots.data_ptr()
        if not _lib.rure_b200_captures_iter_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, d_match_offsets.data_ptr(),
                                                         ptr, cap, byref(total)):
            raise Error(_last_error())
        return total.value

    # ---- diagnostics ------------------------------------------------------------
    def last_stats(self):
        out = (c_double * 13)()
        _lib.rure_b200_last_stats_ex(self._h, out, 13)
        return dict(zip(_STAT_KEYS, list(out)))

    def set_option(self, name, value):
        """Named engine knobs (include/rure_b200.h: rure_b200_set_option)."""
        if not _lib.rure_b200_set_option(self._h, name.encode(), int(value)):
            raise Error(_last_error())

    def set_tuning(self, seg=0, chunk=0, warm=0, block=0, blocks_per_sm=0):
        _lib.rure_b200_set_tuning(self._h, seg, chunk, warm, block, blocks_per_sm)

    def set_stream(self, cuda_stream):
        """Run on the given cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream)."""
        _lib.rure_b200_set_stream(self._h, cuda_stream)

    def set_fuse(self, yes=True):
        _lib.rure_b200_set_fuse(self._h, int(yes))

    def set_tensor_tma(self, yes=True):
        _lib.rure_b200_set_tensor_tma(self._h, int(yes))

    def force_generic(self, yes=True):
        _lib.rure_b200_force_generic(self._h, int(yes))

    def pattern_info(self):
        out = (c_uint64 * 4)()
        _lib.rure_b200_pattern_info(self._h, out)
        return {"min_len": out[0], "max_len": None if out[1] == 2**64 - 1 else out[1], "can_match_empty": bool(out[2]), "has_looks": bool(out[3])}

    def dfa(self, kind):
        """Dense table as numpy arrays (host copy; for tests and tooling)."""
        info = (c_uint32 * 6)()
        if not _lib.rure_b200_dfa_export(self._h, kind, info, None, None, None, None):
            raise Error(_last_error())
        n_states, n_classes, match_lo, mask_words, uniform, raw = list(info)
        trans = np.empty((n_states, n_classes), dtype=np.uint16)
        classes = np.empty(256, dtype=np.uint8)
        start = np.empty(128, dtype=np.uint16)
        masks = np.empty((n_states, mask_words), dtype=np.uint64)
        _lib.rure_b200_dfa_export(self._h, kind, info, trans.ctypes.data, classes.ctypes.data, start.ctypes.data, masks.ctypes.data)
        return {"trans": trans, "classes": classes, "start": start, "masks": masks, "match_lo": match_lo,
                "uniform_start": bool(uniform), "raw_states": raw}


class BytesRegex(_Compiled):
    """`regex::bytes::Regex` (src/re_bytes.rs): haystacks are arbitrary bytes."""
    _only_utf8 = False


class Regex(_Compiled):
    """`regex::Regex` (src/re_unicode.rs): haystacks are str / valid UTF-8; offsets are byte offsets."""
    _only_utf8 = True


class _SetBase:
    _only_utf8 = False

    def last_stats(self):
        out = (c_double * len(_SET_STAT_KEYS))()
        _lib.rure_b200_set_last_stats_ex(self._h, out, len(_SET_STAT_KEYS))
        return dict(zip(_SET_STAT_KEYS, list(out)))

    def set_option(self, name, value):
        """Named engine knobs (include/rure_b200.h: rure_b200_set_set_option), including "set_group_patterns"."""
        if not _lib.rure_b200_set_set_option(self._h, name.encode(), int(value)):
            raise Error(_last_error())

    def groups(self):
        """Pattern groups the set is searched in, as (lo, hi) index ranges: [(0, len(self))] for one product
        automaton (include/rure_b200.h: rure_b200_set_groups)."""
        n = int(_lib.rure_b200_set_groups(self._h, None, 0))
        first = (c_size_t * n)()
        _lib.rure_b200_set_groups(self._h, first, n)
        bounds = list(first) + [len(self)]
        return [(bounds[i], bounds[i + 1]) for i in range(n)]

    def __init__(self, patterns, flags=FLAG_UNICODE, size_limit=10 << 20, dfa_size_limit=2 << 20):
        pats = [p.encode("utf-8") if isinstance(p, str) else bytes(p) for p in patterns]
        self.patterns = list(patterns)
        arr = (c_char_p * max(1, len(pats)))(*pats)
        lens = (c_size_t * max(1, len(pats)))(*[len(p) for p in pats])
        opts = _lib.rure_options_new()
        _lib.rure_options_size_limit(opts, size_limit)
        _lib.rure_options_dfa_size_limit(opts, dfa_size_limit)
        err = _lib.rure_error_new()
        fn = _lib.rure_b200_compile_set_str if self._only_utf8 else _lib.rure_compile_set
        self._h = fn(arr, lens, len(pats), flags, opts, err)
        msg = _lib.rure_error_message(err).decode("utf-8", "replace")
        _lib.rure_error_free(err)
        _lib.rure_options_free(opts)
        if not self._h:
            raise Error(msg)
        self._mw = max(1, (len(pats) + 63) // 64)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and _lib is not None:
            _lib.rure_set_free(h)
            self._h = None

    def __len__(self):
        return int(_lib.rure_set_len(self._h))

    def is_match(self, text, start=0):
        p, n, keep = _buf(text)
        out = c_bool()
        if not _lib.rure_b200_set_is_match(self._h, p, n, start, byref(out)):
            raise Error(_last_error())
        return bool(out.value)

    def matches(self, text, start=0):
        """Indices of the patterns that match somewhere in text (re_set.rs:184-191)."""
        p, n, keep = _buf(text)
        words = self.matches_mask(text, start)  # rure_b200_set_matches_mask reports failures; rure_set_matches aborts
        return [i for i in range(len(self)) if (words[i // 64] >> (i % 64)) & 1]

    def matches_mask(self, text, start=0):
        p, n, keep = _buf(text)
        out = (c_uint64 * self._mw)()
        if not _lib.rure_b200_set_matches_mask(self._h, p, n, start, out):
            raise Error(_last_error())
        return list(out)

    def matches_batch(self, text, offsets):
        """uint64[n_records, mask_words] pattern masks, one row per record."""
        p, n, keep = _buf(text)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = off.size - 1
        out = np.zeros((max(n_rec, 1), self._mw), dtype=np.uint64)
        if not _lib.rure_b200_set_matches_batch(self._h, p, off.ctypes.data, n_rec, out.ctypes.data):
            raise Error(_last_error())
        return out[:n_rec]

    def matches_mask_device(self, d_text, start=0):
        out = (c_uint64 * self._mw)()
        if not _lib.rure_b200_set_matches_device(self._h, d_text.data_ptr(), d_text.numel(), start, out):
            raise Error(_last_error())
        return list(out)

    def set_stream(self, cuda_stream):
        """Run on the given cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream)."""
        _lib.rure_b200_set_set_stream(self._h, cuda_stream)

    def forward_shard_device(self, d_buffer, io):
        """RegexSet::matches over one shard (regex_b200/sharded.py: forward_sharded)."""
        return _forward_shard(_lib.rure_b200_set_matches_shard_device, self._h, d_buffer, io)

    def matches_device(self, d_text, start=0):
        """RegexSet::matches over a device-resident haystack: indices of the matching patterns."""
        words = self.matches_mask_device(d_text, start)
        return [i for i in range(len(self)) if (words[i // 64] >> (i % 64)) & 1]

    def matches_batch_device(self, d_text, d_offsets, d_masks):
        n_rec = d_offsets.numel() - 1
        if not _lib.rure_b200_set_matches_batch_device(self._h, d_text.data_ptr(), d_offsets.data_ptr(), n_rec, d_masks.data_ptr()):
            raise Error(_last_error())

    def set_tuning(self, seg=0, chunk=0, warm=0, block=0, blocks_per_sm=0):
        _lib.rure_b200_set_tuning(self._h, seg, chunk, warm, block, blocks_per_sm)

    def dfa(self, kind=DFA_FWD_UNANCHORED_ALL):
        return _Compiled.dfa(self, kind)


class BytesRegexSet(_SetBase):
    """`regex::bytes::RegexSet` (src/re_set.rs)."""


class RegexSet(_SetBase):
    """`regex::RegexSet` (src/re_set.rs)."""
    _only_utf8 = True


def compiled_with():
    return {"lib": _LIB_PATH, "arch": "sm_100a"}
