"""`aho_corasick::packed` mirrored over libacb200.so (src/packed/api.rs).

Same names and construction contract as the reference -- `Config`, `Builder`, `Searcher`,
`MatchKind`; `Builder.build()` returns None exactly where the reference's does -- and the same
results: non-overlapping leftmost-first / leftmost-longest matches.  On the device there is no
Teddy: the searcher is the K3/K3b kernel pair (fingerprint prefilter + DFA verifier) that also
serves `AhoCorasick`; `Searcher.variant()` reports which Teddy the reference would have run.
"""
from __future__ import annotations

import ctypes as C
import enum

import numpy as np

from . import (MATCH_DTYPE, AhoCorasick, BuildError, DeviceError, Match, _hay_ptr, _i, _lib, _span, _u64, _vp)


class MatchKind(enum.IntEnum):  # src/packed/api.rs:28-46 (values follow include/acb200.h)
    LeftmostFirst = 1
    LeftmostLongest = 2


class _Cfg(C.Structure):
    _fields_ = [("match_kind", C.c_int32), ("force", C.c_int32), ("only_teddy_fat", C.c_int32),
                ("only_teddy_256bit", C.c_int32), ("heuristic_pattern_limits", C.c_int32)]


def _declare(lib):
    """ctypes signatures of the acg_packed_* entry points (include/acb200.h)."""
    lib.acg_packed_build.argtypes = [C.POINTER(C.c_char_p), C.POINTER(_u64), _u64, C.POINTER(_Cfg), C.POINTER(_vp)]
    lib.acg_packed_build_host.argtypes = lib.acg_packed_build.argtypes
    lib.acg_packed_free.argtypes = [_vp]
    lib.acg_packed_free.restype = None
    lib.acg_packed_find_iter.argtypes = [_vp, _vp, _u64, _u64, _u64, _vp, _u64, C.POINTER(_u64)]
    lib.acg_packed_find.argtypes = [_vp, _vp, _u64, _u64, _u64, _vp, C.POINTER(_i)]
    lib.acg_packed_match_kind.argtypes = [_vp]
    for _f in ("acg_packed_minimum_len", "acg_packed_memory_usage", "acg_packed_patterns_len"):
        getattr(lib, _f).argtypes = [_vp]
        getattr(lib, _f).restype = _u64
    lib.acg_packed_searcher_variant.argtypes = [_vp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]


_declare(_lib)


def _opt(v):
    return -1 if v is None else int(bool(v))


class Config:
    """`packed::Config`, src/packed/api.rs:87-230."""

    def __init__(self):
        self._kind = MatchKind.LeftmostFirst
        self._force = 0
        self._fat = None
        self._256 = None
        self._limits = True
        self._host_only = False

    @staticmethod
    def new():
        return Config()

    def builder(self):  # :127
        return Builder(self)

    def match_kind(self, kind):  # :132
        self._kind = MatchKind(kind)
        return self

    def only_teddy(self, yes):  # :143
        self._force = 1 if yes else 0
        return self

    def only_teddy_fat(self, yes):  # :158 (None / False / True)
        self._fat = yes
        return self

    def only_teddy_256bit(self, yes):  # :170
        self._256 = yes
        return self

    def only_rabin_karp(self, yes):  # :181
        self._force = 2 if yes else 0
        return self

    def heuristic_pattern_limits(self, yes):  # :196
        self._limits = bool(yes)
        return self

    def host_only(self, yes=True):
        """Decide and build the tables without touching CUDA (CPU-only checks)."""
        self._host_only = bool(yes)
        return self


class Builder:
    """`packed::Builder`, src/packed/api.rs:232-357."""

    def __init__(self, config: Config | None = None):
        self._cfg = config or Config()
        self._pats = []

    @staticmethod
    def new():
        return Builder()

    def add(self, pattern):  # :303 (the inert rules are applied by the library at build time)
        self._pats.append(pattern.encode() if isinstance(pattern, str) else bytes(pattern))
        return self

    def extend(self, patterns):  # :337
        for p in patterns:
            self.add(p)
        return self

    def len(self):  # :349
        return len(self._pats)

    def minimum_len(self):  # :354
        return min((len(p) for p in self._pats), default=0)

    def build(self):  # :253 -> Searcher or None
        pats = self._pats
        n = len(pats)
        arr = (C.c_char_p * max(n, 1))()
        keep = []
        for i, p in enumerate(pats):
            b = C.create_string_buffer(p, max(len(p), 1))
            keep.append(b)
            arr[i] = C.cast(b, C.c_char_p)
        lens = (_u64 * max(n, 1))(*[len(p) for p in pats])
        c = self._cfg
        cfg = _Cfg(int(c._kind), int(c._force), _opt(c._fat), _opt(c._256), int(c._limits))
        h = _vp()
        fn = _lib.acg_packed_build_host if c._host_only else _lib.acg_packed_build
        rc = fn(arr, lens, n, C.byref(cfg), C.byref(h))
        if rc in (-1, -2, -3):
            raise BuildError(rc)
        if rc:
            raise DeviceError(rc)
        return Searcher(h) if h.value else None


class Searcher:
    """`packed::Searcher`, src/packed/api.rs:396-660."""

    def __init__(self, handle):
        self._h = handle
        self._cap_hint = 4096
        # freed by the library that made it: the CPU dry-run library of tests/emu/ can stand in for
        # `_lib` while searchers made by the other one are still alive
        self._free = _lib.acg_packed_free

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and _lib is not None:
            try:
                self._free(h)
            except Exception:
                pass
            self._h = None

    @staticmethod
    def new(patterns):  # :440
        return Builder().extend(patterns).build()

    @staticmethod
    def config():  # :451
        return Config()

    @staticmethod
    def builder():  # :458
        return Builder()

    _raise = staticmethod(AhoCorasick._raise)

    def find_iter_np(self, hay, span=None):
        def fn(h, ptr, n, s, e, _anchored, out, cap, cnt):
            return _lib.acg_packed_find_iter(h, ptr, n, s, e, out, cap, cnt)
        return AhoCorasick._collect(self, fn, hay, span, 0)

    def find_iter(self, hay, span=None):  # :580 (span=None: the whole haystack, as in the reference)
        r = self.find_iter_np(hay, span)
        return [Match(a, b, c) for a, b, c in zip(r["pid"], r["start"], r["end"])]

    def find_in(self, hay, span):  # :529
        keep, ptr, n = _hay_ptr(hay)
        s, e = _span(span, n)
        out = np.zeros(1, MATCH_DTYPE)
        found = _i()
        rc = _lib.acg_packed_find(self._h, ptr, n, s, e, out.ctypes.data, C.byref(found))
        if rc:
            self._raise(rc)
        if not found.value:
            return None
        return Match(out["pid"][0], out["start"][0], out["end"][0])

    def find(self, hay):  # :491
        return self.find_in(hay, None)

    def match_kind(self):  # :612
        return MatchKind(_lib.acg_packed_match_kind(self._h))

    def minimum_len(self):  # :627
        return _lib.acg_packed_minimum_len(self._h)

    def memory_usage(self):  # :634
        return _lib.acg_packed_memory_usage(self._h)

    def patterns_len(self):
        return _lib.acg_packed_patterns_len(self._h)

    def variant(self):
        """The searcher the reference would run: None for Rabin-Karp, else the Teddy flavour."""
        fat, ml, vb = _i(), _i(), _i()
        if not _lib.acg_packed_searcher_variant(self._h, C.byref(fat), C.byref(ml), C.byref(vb)):
            return None
        return {"fat": bool(fat.value), "mask_len": ml.value, "vector_bytes": vb.value}
