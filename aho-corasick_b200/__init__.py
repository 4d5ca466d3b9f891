"""aho_corasick_b200 -- host-side mirror of the reference's search API over libacb200.so.

The names, argument meaning and error behaviour follow BurntSushi/aho-corasick 1.1.3
(`AhoCorasick`, `AhoCorasickBuilder`, `MatchKind`, `StartKind`, `AhoCorasickKind`, `Match`,
`find_iter`, `find_overlapping_iter`, `try_*`; src/ahocorasick.rs, src/lib.rs:239-251), so the
parity tests read like the reference's own.  Everything that touches a haystack goes through the
C ABI (include/acb200.h) into hand-written sm_100a kernels; there is no CPU search path here.
Python is test/bench glue only: the product is the shared library.
"""
from __future__ import annotations

import ctypes as C
import enum
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "libacb200.so"


class NativeLibraryMissing(ImportError):
    pass


def _load():
    if not _LIB_PATH.exists():
        raise NativeLibraryMissing(
            f"{_LIB_PATH} is missing: build it with `python aho-corasick_b200/build.py` "
            "(nvcc, sm_100a). There is no fallback implementation.")
    return C.CDLL(str(_LIB_PATH))


_lib = _load()


class MatchKind(enum.IntEnum):  # src/util/search.rs:1052
    Standard = 0
    LeftmostFirst = 1
    LeftmostLongest = 2


class StartKind(enum.IntEnum):  # src/util/search.rs:1133
    Unanchored = 0
    Anchored = 1
    Both = 2


class AhoCorasickKind(enum.IntEnum):  # src/ahocorasick.rs:2624
    NoncontiguousNFA = 1
    ContiguousNFA = 2
    DFA = 3


class Anchored(enum.IntEnum):  # src/util/search.rs:784
    No = 0
    Yes = 1


class Engine(enum.IntEnum):
    Auto = 0
    Walk = 1
    Prefilter = 2
    Sequential = 3


E_OVERFLOW = -21


class BuildError(Exception):  # src/util/error.rs:23-49
    def __init__(self, code):
        super().__init__(_lib.acg_strerror(code).decode())
        self.code = code


class MatchError(Exception):  # src/util/error.rs:140-223
    def __init__(self, code):
        super().__init__(_lib.acg_strerror(code).decode())
        self.code = code

    @property
    def kind(self):
        return {-10: "InvalidInputAnchored", -11: "InvalidInputUnanchored", -12: "UnsupportedStream",
                -13: "UnsupportedOverlapping", -14: "UnsupportedEmpty"}.get(self.code, "Boundary")


class DeviceError(RuntimeError):
    def __init__(self, code):
        super().__init__(_lib.acg_strerror(code).decode())
        self.code = code


class _BuildOpts(C.Structure):
    _fields_ = [("match_kind", C.c_int32), ("start_kind", C.c_int32),
                ("ascii_case_insensitive", C.c_int32), ("byte_classes", C.c_int32),
                ("prefilter", C.c_int32), ("kind", C.c_int32), ("dense_depth", C.c_int64)]


class _Desc(C.Structure):
    _fields_ = [("trans", C.POINTER(C.c_uint32)), ("trans_len", C.c_uint64),
                ("stride2", C.c_uint32), ("alphabet_len", C.c_uint32),
                ("byte_classes", C.c_uint8 * 256),
                ("max_special_id", C.c_uint32), ("max_match_id", C.c_uint32),
                ("start_unanchored_id", C.c_uint32), ("start_anchored_id", C.c_uint32),
                ("match_offsets", C.POINTER(C.c_uint32)), ("match_pids", C.POINTER(C.c_uint32)),
                ("pattern_lens", C.POINTER(C.c_uint32)), ("n_patterns", C.c_uint32),
                ("match_kind", C.c_uint32), ("start_kind", C.c_uint32), ("prefilter_kind", C.c_uint32),
                ("min_pattern_len", C.c_uint64), ("max_pattern_len", C.c_uint64)]


class _Stats(C.Structure):
    _fields_ = [("engine", C.c_int32), ("launches", C.c_int32), ("candidates", C.c_uint64),
                ("raw_matches", C.c_uint64), ("scan_ms", C.c_float), ("order_ms", C.c_float),
                ("h2d_ms", C.c_float), ("d2h_ms", C.c_float)]


MATCH_DTYPE = np.dtype([("pid", "<u4"), ("_pad", "<u4"), ("start", "<u8"), ("end", "<u8")])

_vp, _u64, _i = C.c_void_p, C.c_uint64, C.c_int


def _declare(lib):
    """ctypes signatures of the C ABI (include/acb200.h)."""
    lib.acg_strerror.restype = C.c_char_p
    lib.acg_strerror.argtypes = [_i]
    lib.acg_build.argtypes = [C.POINTER(C.c_char_p), C.POINTER(_u64), _u64, C.POINTER(_BuildOpts), C.POINTER(_vp)]
    lib.acg_build_host.argtypes = lib.acg_build.argtypes
    lib.acg_build_on_device.argtypes = lib.acg_build.argtypes
    lib.acg_dfa_create.argtypes = [C.POINTER(_Desc), C.POINTER(_vp)]
    lib.acg_dfa_free.argtypes = [_vp]
    lib.acg_dfa_free.restype = None
    lib.acg_dfa_table.argtypes = [_vp, C.POINTER(_Desc)]
    for _f in ("acg_dfa_state_len", "acg_patterns_len", "acg_min_pattern_len", "acg_max_pattern_len",
               "acg_memory_usage"):
        getattr(lib, _f).argtypes = [_vp]
        getattr(lib, _f).restype = _u64
    for _f in ("acg_kind", "acg_match_kind", "acg_start_kind", "acg_prefilter_kind", "acg_last_engine"):
        getattr(lib, _f).argtypes = [_vp]
    lib.acg_packed_variant.argtypes = [_vp, C.POINTER(_i), C.POINTER(_i)]
    lib.acg_set_engine.argtypes = [_vp, _i]
    lib.acg_last_stats.argtypes = [_vp, C.POINTER(_Stats)]
    lib.acg_find_overlapping.argtypes = [_vp, _vp, _u64, _u64, _u64, _i, _vp, _u64, C.POINTER(_u64)]
    lib.acg_find_iter.argtypes = lib.acg_find_overlapping.argtypes
    lib.acg_find.argtypes = [_vp, _vp, _u64, _u64, _u64, _i, _i, _vp, C.POINTER(_i)]
    lib.acg_find_overlapping_dev.argtypes = [_vp, _vp, _u64, _u64, _u64, _vp, _u64, C.POINTER(_u64),
                                              C.POINTER(C.c_float)]
    lib.acg_find_iter_dev.argtypes = lib.acg_find_overlapping_dev.argtypes
    lib.acg_count_overlapping_dev.argtypes = [_vp, _vp, _u64, _u64, _u64, C.POINTER(_u64), C.POINTER(_u64),
                                               C.POINTER(C.c_float)]
    lib.acg_find_overlapping_devout.argtypes = [_vp, _vp, _u64, _u64, _u64, _u64, _u64, _vp, _u64,
                                                 C.POINTER(_u64), C.POINTER(C.c_float)]
    lib.acg_device_count.argtypes = []
    # multi-GPU (include/acb200.h, SURVEY.md section 8e)
    lib.acg_comm_unique_id.argtypes = [_vp]
    lib.acg_comm_init.argtypes = [_vp, _i, _i, C.POINTER(_vp)]
    lib.acg_comm_free.argtypes = [_vp]
    lib.acg_comm_free.restype = None
    lib.acg_comm_rank.argtypes = [_vp]
    lib.acg_comm_size.argtypes = [_vp]
    lib.acg_comm_transport.argtypes = [_vp]
    lib.acg_shard_plan.argtypes = [_u64, _u64, _i, _i, _u64, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64)]
    lib.acg_find_overlapping_sharded.argtypes = [_vp, _vp, _vp, _i, _u64, _u64, _u64, _u64, C.POINTER(_vp),
                                                  C.POINTER(_u64), _vp, _u64, _vp]
    lib.acg_find_overlapping_sharded_begin.argtypes = [_vp, _vp, _vp, _i, _u64, _u64, _u64, _u64, C.POINTER(_i)]
    lib.acg_find_overlapping_sharded_wait.argtypes = [_vp, _i, C.POINTER(_vp), C.POINTER(_u64), _vp, _u64, _vp]
    lib.acg_comm_mark.argtypes = [_vp, _i]
    lib.acg_comm_mark_elapsed_ms.argtypes = [_vp, C.POINTER(C.c_float)]
    lib.acg_comm_fetch.argtypes = [_vp, _vp, _u64, C.POINTER(_u64)]
    lib.acg_comm_fetch_view.argtypes = [_vp, C.POINTER(_vp), C.POINTER(_u64)]
    lib.acg_comm_checksum.argtypes = [_vp, C.POINTER(_u64), C.POINTER(_u64)]


_declare(_lib)


def device_count() -> int:
    return _lib.acg_device_count()


class Match:
    """`Match`, src/util/search.rs:825-830."""
    __slots__ = ("_pid", "_start", "_end")

    def __init__(self, pid, start, end):
        self._pid, self._start, self._end = int(pid), int(start), int(end)

    def pattern(self):
        return self._pid

    def start(self):
        return self._start

    def end(self):
        return self._end

    def span(self):
        return (self._start, self._end)

    def is_empty(self):
        return self._start == self._end

    def as_tuple(self):
        return (self._pid, self._start, self._end)

    def __eq__(self, o):
        return isinstance(o, Match) and self.as_tuple() == o.as_tuple()

    def __repr__(self):
        return f"Match(pattern={self._pid}, span={self._start}..{self._end})"


def _hay_ptr(hay):
    """(keepalive, address, length) of a bytes-like / contiguous uint8 ndarray haystack."""
    if isinstance(hay, np.ndarray):
        if hay.dtype != np.uint8 or not hay.flags["C_CONTIGUOUS"]:
            raise TypeError("haystack ndarray must be contiguous uint8")
        return hay, hay.ctypes.data, hay.size
    if isinstance(hay, str):
        hay = hay.encode()
    arr = np.frombuffer(bytes(hay) if not isinstance(hay, (bytes, bytearray, memoryview)) else hay, dtype=np.uint8)
    return arr, arr.ctypes.data if arr.size else 0, arr.size


def _span(span, n):
    if span is None:
        return 0, n
    return int(span[0]), int(span[1])


class Input:
    """`Input`, src/util/search.rs:60-720: a haystack with a span, an anchored mode and the
    `earliest` flag.  Every search method accepts either a plain haystack (with keyword arguments)
    or an `Input`."""
    __slots__ = ("_hay", "_n", "_start", "_end", "_anchored", "_earliest")

    def __init__(self, haystack):  # Input::new, :93
        keep, _, n = _hay_ptr(haystack)
        self._hay, self._n = keep, n
        self._start, self._end = 0, n
        self._anchored, self._earliest = Anchored.No, False

    new = staticmethod(lambda haystack: Input(haystack))

    def clone(self):
        c = Input.__new__(Input)
        for k in Input.__slots__:
            setattr(c, k, getattr(self, k))
        return c

    # builder-style setters (consume and return, :142-310)
    def span(self, span):
        self.set_span(span)
        return self

    def range(self, rng):
        self.set_range(rng)
        return self

    def anchored(self, mode):
        self.set_anchored(mode)
        return self

    def earliest(self, yes):
        self.set_earliest(yes)
        return self

    # setters (:332-480)
    def set_span(self, span):
        start, end = int(span[0]), int(span[1])
        # the reference panics on an invalid span (:335-341)
        if not (0 <= start and end <= self._n and start <= end + 1):
            raise ValueError(f"invalid span ({start}, {end}) for haystack of length {self._n}")
        self._start, self._end = start, end

    def set_range(self, rng):
        if isinstance(rng, (range, slice)):
            if rng.step not in (None, 1):
                raise ValueError("ranges must have step 1")
            start = 0 if rng.start is None else rng.start
            end = self._n if rng.stop is None else rng.stop
            rng = (start, end)
        self.set_span(rng)

    def set_start(self, start):
        self.set_span((start, self._end))

    def set_end(self, end):
        self.set_span((self._start, end))

    def set_anchored(self, mode):
        self._anchored = Anchored(mode)

    def set_earliest(self, yes):
        self._earliest = bool(yes)

    # getters (:493-630)
    def haystack(self):
        return self._hay

    def start(self):
        return self._start

    def end(self):
        return self._end

    def get_span(self):
        return (self._start, self._end)

    def get_range(self):
        return range(self._start, self._end)

    def get_anchored(self):
        return self._anchored

    def get_earliest(self):
        return self._earliest

    def is_done(self):  # :627
        return self._start > self._end


class OverlappingState:
    """`OverlappingState`, src/automaton.rs:782-840: the cursor of a resumable overlapping search.
    The device scan is eager, so the state holds the ordered match list of the search it was first
    used with and hands out one match per `try_find_overlapping` call -- the same sequence the
    reference's state machine produces.  As in the reference, a state must be reused only with the
    same automaton and input."""
    __slots__ = ("_matches", "_next", "_mat")

    def __init__(self):
        self._matches = None
        self._next = 0
        self._mat = None

    @staticmethod
    def start():  # :817
        return OverlappingState()

    def get_match(self):  # :829
        return self._mat


class AhoCorasickBuilder:
    """`AhoCorasickBuilder`, src/ahocorasick.rs:2135-2617 (same knobs, same defaults)."""

    def __init__(self):
        self._o = dict(match_kind=MatchKind.Standard, start_kind=StartKind.Unanchored,
                       ascii_case_insensitive=False, byte_classes=True, prefilter=True, kind=None,
                       dense_depth=3)
        self._host_only = False
        self._device_fill = False

    def match_kind(self, kind):
        self._o["match_kind"] = MatchKind(kind)
        return self

    def start_kind(self, kind):
        self._o["start_kind"] = StartKind(kind)
        return self

    def ascii_case_insensitive(self, yes):
        self._o["ascii_case_insensitive"] = bool(yes)
        return self

    def kind(self, kind):
        self._o["kind"] = None if kind is None else AhoCorasickKind(kind)
        return self

    def prefilter(self, yes):
        self._o["prefilter"] = bool(yes)
        return self

    def dense_depth(self, depth):
        self._o["dense_depth"] = int(depth)
        return self

    def byte_classes(self, yes):
        self._o["byte_classes"] = bool(yes)
        return self

    def host_only(self, yes=True):
        """Build the tables without touching CUDA (table-parity checks on CPU-only machines)."""
        self._host_only = bool(yes)
        return self

    def device_fill(self, yes=True):
        """Produce the dense transition table on the GPU (acg_build_on_device) instead of building it on
        the host and copying it over; same table, same results."""
        self._device_fill = bool(yes)
        return self

    def build(self, patterns):
        pats = [p.encode() if isinstance(p, str) else bytes(p) for p in patterns]
        n = len(pats)
        # one contiguous buffer + a pointer per pattern (a ctypes object per pattern costs ~3 us each:
        # a third of a second for the 100 000 patterns of BASELINE config 5)
        lens_np = np.fromiter((len(p) for p in pats), dtype=np.uint64, count=n) if n else np.zeros(1, np.uint64)
        blob = np.frombuffer(b"".join(pats) + b"\0", dtype=np.uint8)
        offs = np.zeros(max(n, 1), dtype=np.uint64)
        if n > 1:
            np.cumsum(lens_np[:-1], out=offs[1:n])
        ptrs = (offs + np.uint64(blob.ctypes.data)).astype(np.uint64)
        arr = ptrs.ctypes.data_as(C.POINTER(C.c_char_p))
        lens = lens_np.ctypes.data_as(C.POINTER(_u64))
        keep = (blob, ptrs, lens_np)
        o = self._o
        opts = _BuildOpts(int(o["match_kind"]), int(o["start_kind"]), int(o["ascii_case_insensitive"]),
                          int(o["byte_classes"]), int(o["prefilter"]), int(o["kind"] or 0), o["dense_depth"])
        h = _vp()
        fn = _lib.acg_build_host if self._host_only else (_lib.acg_build_on_device if self._device_fill else _lib.acg_build)
        rc = fn(arr, lens, n, C.byref(opts), C.byref(h))
        if rc in (-1, -2, -3):
            raise BuildError(rc)
        if rc:
            raise DeviceError(rc)
        return AhoCorasick(h)


class AhoCorasick:
    """`AhoCorasick`, src/ahocorasick.rs:177-2082 (search surface only; replace/stream are out of scope)."""

    def __init__(self, handle):
        self._h = handle
        self._cap_hint = 4096  # output-buffer sizing for the two-call overflow protocol
        # freed by the library that made it: the CPU dry-run library of tests/emu/ can stand in for
        # `_lib` while handles made by the other one are still alive
        self._free = _lib.acg_dfa_free

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and _lib is not None:
            try:
                self._free(h)
            except Exception:
                pass
            self._h = None

    @staticmethod
    def new(patterns):  # src/ahocorasick.rs:243
        return AhoCorasickBuilder().build(patterns)

    @staticmethod
    def builder():  # src/ahocorasick.rs:268
        return AhoCorasickBuilder()

    @staticmethod
    def from_dfa_tables(t: dict):
        """Adopt a DFA built elsewhere (what a Rust -sys shim does): acg_dfa_create."""
        d = _Desc()
        keep = {}

        def arr(name, dtype=np.uint32):
            a = np.ascontiguousarray(t[name], dtype=dtype)
            keep[name] = a
            return a.ctypes.data_as(C.POINTER(C.c_uint32))
        d.trans = arr("trans")
        d.trans_len = keep["trans"].size
        d.stride2, d.alphabet_len = int(t["stride2"]), int(t["alphabet_len"])
        bc = np.ascontiguousarray(t["byte_classes"], dtype=np.uint8)
        C.memmove(d.byte_classes, bc.ctypes.data, 256)
        for k in ("max_special_id", "max_match_id", "start_unanchored_id", "start_anchored_id"):
            setattr(d, k, int(t[k]))
        d.match_offsets = arr("match_offsets")
        d.match_pids = arr("match_pids")
        d.pattern_lens = arr("pattern_lens")
        d.n_patterns = keep["pattern_lens"].size
        d.match_kind = int(t["match_kind"])
        d.start_kind = int(t.get("start_kind", 0))
        d.prefilter_kind = int(t.get("prefilter_kind", 0))
        d.min_pattern_len, d.max_pattern_len = int(t["min_pattern_len"]), int(t["max_pattern_len"])
        h = _vp()
        rc = _lib.acg_dfa_create(C.byref(d), C.byref(h))
        if rc:
            raise DeviceError(rc)
        return AhoCorasick(h)

    # ---- getters (src/ahocorasick.rs:1867-2021) ----
    def kind(self):
        return AhoCorasickKind(_lib.acg_kind(self._h))

    def start_kind(self):
        return StartKind(_lib.acg_start_kind(self._h))

    def match_kind(self):
        return MatchKind(_lib.acg_match_kind(self._h))

    def min_pattern_len(self):
        return _lib.acg_min_pattern_len(self._h)

    def max_pattern_len(self):
        return _lib.acg_max_pattern_len(self._h)

    def patterns_len(self):
        return _lib.acg_patterns_len(self._h)

    def memory_usage(self):
        return _lib.acg_memory_usage(self._h)

    def prefilter_kind(self):
        return _lib.acg_prefilter_kind(self._h)

    def packed_variant(self):
        fat, ml = _i(), _i()
        if not _lib.acg_packed_variant(self._h, C.byref(fat), C.byref(ml)):
            return None
        return {"fat": bool(fat.value), "mask_len": ml.value}

    def state_len(self):
        return _lib.acg_dfa_state_len(self._h)

    def tables(self) -> dict:
        d = _Desc()
        rc = _lib.acg_dfa_table(self._h, C.byref(d))  # fetches the table of a device-filled handle
        if rc:
            raise DeviceError(rc)
        nms = (d.max_match_id >> d.stride2) - 1

        def arr(ptr, n):
            return np.ctypeslib.as_array(ptr, (n,)).copy() if n and ptr else np.zeros(0, np.uint32)
        offs = arr(d.match_offsets, nms + 1)
        tot = int(offs[-1])
        return {
            "trans": arr(d.trans, d.trans_len),
            "stride2": d.stride2, "alphabet_len": d.alphabet_len,
            "byte_classes": np.frombuffer(bytes(d.byte_classes), dtype=np.uint8).copy(),
            "max_special_id": d.max_special_id, "max_match_id": d.max_match_id,
            "start_unanchored_id": d.start_unanchored_id, "start_anchored_id": d.start_anchored_id,
            "match_offsets": offs,
            "match_pids": arr(d.match_pids, tot),
            "pattern_lens": arr(d.pattern_lens, d.n_patterns),
            "match_kind": d.match_kind, "start_kind": d.start_kind, "prefilter_kind": d.prefilter_kind,
            "min_pattern_len": d.min_pattern_len, "max_pattern_len": d.max_pattern_len,
            "state_len": _lib.acg_dfa_state_len(self._h),
        }

    # ---- engine control / stats (device-side knobs that do not exist in the reference) ----
    def set_engine(self, engine):
        rc = _lib.acg_set_engine(self._h, int(engine))
        if rc:
            raise DeviceError(rc)
        return self

    def last_stats(self) -> dict:
        s = _Stats()
        _lib.acg_last_stats(self._h, C.byref(s))
        return {k: getattr(s, k) for k, _ in _Stats._fields_}

    # ---- searches ----
    @staticmethod
    def _raise(rc):
        if -14 <= rc <= -10:
            raise MatchError(rc)
        if rc == -20:
            raise ValueError("invalid span for haystack")  # the reference panics (search.rs:332-343)
        raise DeviceError(rc)

    def _collect(self, fn, hay, span, anchored):
        if isinstance(hay, Input):
            hay, span, anchored = hay.haystack(), hay.get_span(), hay.get_anchored()
        keep, ptr, n = _hay_ptr(hay)
        s, e = _span(span, n)
        # room for one match per 256 haystack bytes from the start (the device sizes its own tuple buffer the
        # same way): an overflow retry repeats the whole copy + scan, so it should be the exception
        cap = max(self._cap_hint, max(e - s, 0) // 256 + 64)
        while True:
            out = np.empty(cap, MATCH_DTYPE)
            cnt = _u64()
            rc = fn(self._h, ptr, n, s, e, int(anchored), out.ctypes.data, cap, C.byref(cnt))
            if rc == E_OVERFLOW:  # the call reports the required count: retry once with room to spare
                cap = int(cnt.value) + int(cnt.value) // 8 + 64
                self._cap_hint = max(self._cap_hint, cap)
                continue
            if rc:
                self._raise(rc)
            return out[: cnt.value]

    def try_find_iter_np(self, hay, span=None, anchored=Anchored.No):
        return self._collect(_lib.acg_find_iter, hay, span, anchored)

    def try_find_overlapping_iter_np(self, hay, span=None, anchored=Anchored.No):
        return self._collect(_lib.acg_find_overlapping, hay, span, anchored)

    def try_find_iter(self, hay, span=None, anchored=Anchored.No):  # src/ahocorasick.rs:1275
        r = self.try_find_iter_np(hay, span, anchored)
        return [Match(a, b, c) for a, b, c in zip(r["pid"], r["start"], r["end"])]

    def try_find_overlapping_iter(self, hay, span=None, anchored=Anchored.No):  # :1350
        r = self.try_find_overlapping_iter_np(hay, span, anchored)
        return [Match(a, b, c) for a, b, c in zip(r["pid"], r["start"], r["end"])]

    def try_find_overlapping(self, hay, state: OverlappingState, span=None, anchored=Anchored.No):
        """`try_find_overlapping`, src/ahocorasick.rs:1184: advance `state` to the next overlapping
        match (or to None).  Errors are the ones of try_find_overlapping_iter (src/automaton.rs
        :397-423) and are reported on every call, as in the reference."""
        if state._matches is None:
            state._matches = self.try_find_overlapping_iter(hay, span, anchored)
            state._next = 0
        if state._next < len(state._matches):
            state._mat = state._matches[state._next]
            state._next += 1
        else:
            state._mat = None

    find_overlapping = try_find_overlapping  # :470

    find_iter = try_find_iter  # :562 (the infallible versions panic where these raise)
    find_overlapping_iter = try_find_overlapping_iter  # :609

    def try_find(self, hay, span=None, anchored=Anchored.No, earliest=False):  # :1021
        if isinstance(hay, Input):
            hay, span, anchored, earliest = hay.haystack(), hay.get_span(), hay.get_anchored(), hay.get_earliest()
        keep, ptr, n = _hay_ptr(hay)
        s, e = _span(span, n)
        out = np.zeros(1, MATCH_DTYPE)
        found = _i()
        rc = _lib.acg_find(self._h, ptr, n, s, e, int(anchored), int(earliest), out.ctypes.data, C.byref(found))
        if rc:
            self._raise(rc)
        if not found.value:
            return None
        return Match(out["pid"][0], out["start"][0], out["end"][0])

    find = try_find  # :404

    def is_match(self, hay, span=None):  # :311
        # The reference asks for the earliest match; only existence is reported, and a match exists
        # under `earliest` iff one exists without it, so leftmost automata stay on the windowed
        # device scan instead of the single-lane engine.
        earliest = self.match_kind() == MatchKind.Standard
        if isinstance(hay, Input):
            return self.try_find(hay.clone().earliest(earliest)) is not None
        return self.try_find(hay, span, earliest=earliest) is not None

    # ---- replace / stream: host-side glue over find_iter, as in the reference -------------------
    @staticmethod
    def _is_char_boundary(view, n, i):
        """`str::is_char_boundary` on UTF-8 bytes."""
        if i == 0 or i == n:
            return True
        return i < n and (view[i] & 0xC0) != 0x80

    @staticmethod
    def _splice(view, n, matches, dst: bytearray, replace_with, char_boundaries=False):
        """The loop of `try_replace_all_with{,_bytes}`, src/automaton.rs:498-550, over an already
        materialised match list.  With `char_boundaries` (the `&str` flavour) matches that split a
        UTF-8 code point are skipped (:514-518)."""
        last = 0
        for m in matches:
            if char_boundaries and not (AhoCorasick._is_char_boundary(view, n, m.start())
                                        and AhoCorasick._is_char_boundary(view, n, m.end())):
                continue
            dst += bytes(view[last:m.start()])
            last = m.end()
            if not replace_with(m, bytes(view[m.start():m.end()]), dst):
                break
        dst += bytes(view[last:])

    def try_replace_all_with(self, hay, dst: bytearray, replace_with):
        """`try_replace_all_with_bytes`, src/automaton.rs:525-550: `replace_with(match, matched
        bytes, dst) -> bool`; returning False stops the replacement after that match."""
        keep, ptr, n = _hay_ptr(hay)
        view = memoryview(keep).cast("B") if n else b""
        self._splice(view, n, self.try_find_iter(keep), dst, replace_with)

    def _replacements(self, replace_with):
        if len(replace_with) != self.patterns_len():
            raise ValueError("replace_all requires a replacement for every pattern in the automaton")
        return [r.encode() if isinstance(r, str) else bytes(r) for r in replace_with]

    def try_replace_all_bytes(self, hay, replace_with):  # src/automaton.rs:457-480
        reps = self._replacements(replace_with)
        dst = bytearray()

        def put(m, _, out):
            out += reps[m.pattern()]
            return True
        self.try_replace_all_with(hay, dst, put)
        return bytes(dst)

    def try_replace_all(self, hay: str, replace_with):  # src/automaton.rs:433-455 -> :498-523
        reps = self._replacements(replace_with)
        keep, ptr, n = _hay_ptr(hay.encode())
        view = memoryview(keep).cast("B") if n else b""
        dst = bytearray()

        def put(m, _, out):
            out += reps[m.pattern()]
            return True
        self._splice(view, n, self.try_find_iter(keep), dst, put, char_boundaries=True)
        return dst.decode()

    replace_all = try_replace_all                # src/ahocorasick.rs:651
    replace_all_bytes = try_replace_all_bytes    # :693
    replace_all_with = try_replace_all_with      # :834 (bytes flavour)

    def _stream_chunks(self, rdr, chunk_bytes):
        """`StreamChunkIter`, src/automaton.rs:1059-1256: the stream as an alternation of
        ("bytes", data) for text between matches and ("match", Match, matched bytes), offsets
        relative to the start of the stream.  Like the reference it is limited to
        MatchKind::Standard without empty patterns (:1087-1103), and like the reference's roll buffer
        (src/util/buffer.rs) only max_pattern_len-1 bytes are carried from one device scan to the
        next: a match that straddles a block boundary starts no earlier than that."""
        if self.match_kind() != MatchKind.Standard:
            raise MatchError(-12)
        if self.patterns_len() and self.min_pattern_len() == 0:
            raise MatchError(-14)
        back = max(self.max_pattern_len() - 1, 0)
        carry = b""
        base = 0          # stream offset of carry[0]
        cursor = 0        # stream offset where the iterator restarts
        emitted = 0       # stream offset up to which chunks have been yielded
        while True:
            block = rdr.read(chunk_bytes)
            if not block:
                break
            buf = np.frombuffer(carry + bytes(block), dtype=np.uint8)
            r = self.try_find_iter_np(buf, span=(cursor - base, buf.size))
            for pid, s, e in zip(r["pid"].tolist(), r["start"].tolist(), r["end"].tolist()):
                if base + s > emitted:
                    yield ("bytes", buf[emitted - base:s].tobytes())
                yield ("match", Match(pid, base + s, base + e), buf[s:e].tobytes())
                emitted = base + e
            if len(r):
                cursor = base + int(r["end"][-1])
            keep_from = max(cursor, base + buf.size - back)
            if keep_from > emitted:  # these bytes can no longer be part of a match
                yield ("bytes", buf[emitted - base:keep_from - base].tobytes())
                emitted = keep_from
            carry = buf[keep_from - base:].tobytes()
            base = keep_from
            cursor = max(cursor, base)
        if emitted - base < len(carry):
            yield ("bytes", carry[emitted - base:])

    def try_stream_find_iter(self, rdr, chunk_bytes=64 << 20):
        """`try_stream_find_iter`, src/ahocorasick.rs:1677: matches of a byte stream (anything with
        .read(n)); equals find_iter over the concatenated stream."""
        for chunk in self._stream_chunks(rdr, chunk_bytes):
            if chunk[0] == "match":
                yield chunk[1]

    stream_find_iter = try_stream_find_iter      # :906

    def try_stream_replace_all_with(self, rdr, wtr, replace_with, chunk_bytes=64 << 20):
        """`try_stream_replace_all_with`, src/ahocorasick.rs:1807 -> src/automaton.rs:601-636:
        `replace_with(match, matched bytes, wtr)` writes the replacement; text between matches is
        copied through as soon as it can no longer be part of a match."""
        for chunk in self._stream_chunks(rdr, chunk_bytes):
            if chunk[0] == "bytes":
                wtr.write(chunk[1])
            else:
                replace_with(chunk[1], chunk[2], wtr)

    def try_stream_replace_all(self, rdr, wtr, replace_with, chunk_bytes=64 << 20):  # :1751
        if len(replace_with) != self.patterns_len():
            raise ValueError("stream_replace_all requires a replacement for every pattern in the automaton")
        reps = [r.encode() if isinstance(r, str) else bytes(r) for r in replace_with]
        self.try_stream_replace_all_with(rdr, wtr, lambda m, _, w: w.write(reps[m.pattern()]), chunk_bytes)

    stream_replace_all = try_stream_replace_all            # :964
    stream_replace_all_with = try_stream_replace_all_with  # :1007

    # ---- device-resident haystack (torch tensor / raw pointer), for the roofline measurement ----
    def find_overlapping_iter_dev_np(self, dev_ptr, hay_len, span=None):
        s, e = _span(span, hay_len)
        cap = max(self._cap_hint, 1 << 16)
        while True:
            out = np.empty(cap, MATCH_DTYPE)
            cnt, ms = _u64(), C.c_float()
            rc = _lib.acg_find_overlapping_dev(self._h, dev_ptr, hay_len, s, e, out.ctypes.data, cap,
                                               C.byref(cnt), C.byref(ms))
            if rc == E_OVERFLOW:
                cap = int(cnt.value) + int(cnt.value) // 8 + 64
                self._cap_hint = max(self._cap_hint, cap)
                continue
            if rc:
                self._raise(rc)
            return out[: cnt.value], ms.value

    def find_iter_dev_np(self, dev_ptr, hay_len, span=None):
        s, e = _span(span, hay_len)
        cap = max(self._cap_hint, 1 << 16)
        while True:
            out = np.empty(cap, MATCH_DTYPE)
            cnt, ms = _u64(), C.c_float()
            rc = _lib.acg_find_iter_dev(self._h, dev_ptr, hay_len, s, e, out.ctypes.data, cap,
                                        C.byref(cnt), C.byref(ms))
            if rc == E_OVERFLOW:
                cap = int(cnt.value) + int(cnt.value) // 8 + 64
                self._cap_hint = max(self._cap_hint, cap)
                continue
            if rc:
                self._raise(rc)
            return out[: cnt.value], ms.value

    def find_overlapping_devout(self, dev_ptr, hay_len, span, min_end, offset_add, out_ptr, cap):
        """Ordered matches stay on the device (acg_match records at out_ptr). Returns (n, kernel_ms);
        raises OverflowError(needed) if cap is too small."""
        s, e = _span(span, hay_len)
        cnt, ms = _u64(), C.c_float()
        rc = _lib.acg_find_overlapping_devout(self._h, dev_ptr, hay_len, s, e, min_end, offset_add,
                                              out_ptr, cap, C.byref(cnt), C.byref(ms))
        if rc == E_OVERFLOW:
            raise OverflowError(int(cnt.value))
        if rc:
            self._raise(rc)
        return int(cnt.value), ms.value

    def count_overlapping_dev(self, dev_ptr, hay_len, span=None):
        s, e = _span(span, hay_len)
        cnt, fnv, ms = _u64(), _u64(), C.c_float()
        rc = _lib.acg_count_overlapping_dev(self._h, dev_ptr, hay_len, s, e, C.byref(cnt), C.byref(fnv),
                                            C.byref(ms))
        if rc:
            self._raise(rc)
        return cnt.value, fnv.value, ms.value
