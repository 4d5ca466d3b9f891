"""Every prefilter kernel instantiation, the byte-set scan and the brute-force path on the device,
pinned by name (the plan each case claims is read back through acg_debug_prefilter_plan) and compared
tuple for tuple, order included, with the CPU oracle.

launch_prefilter (csrc/acb_prefilter.cu) picks prefilter_kernel from a table indexed by
[MODE][masked][tile distribution][variant]: MODE 0 (every occurrence: find_overlapping_iter, and
Standard find_iter with first_only) / MODE 1 (best match per start: leftmost find_iter); masked =
case folding or k < 4; tiles static (ACG_EXP_STATIC_TILES = 32) / per-CTA counter (default) / global
super-tiles (ACG_EXP_GLOBAL_TILES = 16); variant stride 1 / stride 1 + dense / stride 2 narrow /
stride 2 wide.  All 48 are reachable from plans derive_metadata makes, and the case table below
reaches all of them (test_case_table_covers_every_instantiation checks that without a GPU).

Beyond the matrix: guard bytes around the haystack and the span at every pointer phase, ragged
sizes on every engine, the host-copy paths (pageable with and without the staging ring, page-locked,
many pipeline chunks, matches across every chunk boundary) and concurrent searches on shared handles.

Under the CPU dry run (ACB_EMULATE=1, tests/emu) the same cases run at reduced sizes; the
page-locked cases need a device and skip there."""
import ctypes
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import aho_corasick_b200 as ab
import oracle_py as O
from aho_corasick_b200 import workload as W
from test_gpu_parity import assert_np_equal, to_device
from test_prefilter_plan import plan_of, set_experiment

ON_GPU = torch.cuda.is_available()
MiB = 1 << 20
# The dry run executes one CTA at a time with CUDA threads as fibers: the same cases at 1/64 size.
SCALE = 1.0 if ON_GPU else 1 / 64
PREFILTER = int(ab.Engine.Prefilter)


def scaled(nbytes):
    return max(int(nbytes * SCALE) // 16 * 16, 64 << 10)


# ---- pattern sets ----------------------------------------------------------------------------------
def _k3_set():
    p = W.make_patterns(300, 31)
    return [x[:3] for x in p[:150]] + p[150:]


PATTERN_SETS = {
    "cfg2": lambda: W.make_patterns(5000, 0xAC5000),                            # stride 2 narrow (BASELINE 2 / 3)
    "cfg4": lambda: W.make_patterns(50, 0xAC0050),                              # stride 2 wide (BASELINE 4)
    "dense": lambda: W.make_patterns(20000, 0xAC1000),                          # > 8192 fingerprints: dense
    "k4_ap": lambda: W.make_patterns(3000, 13, lo=4, hi=8, alphabet=(0x61, 0x70)),  # common 3-grams: stride 1
    "k3": _k3_set,                                                              # 3-byte patterns: k = 3
    "brute": lambda: W.make_patterns(300, 7, lo=4, hi=8, alphabet=(0x61, 0x64)),    # unselective: brute force
    "bytes_m0": lambda: [b"Quartz", b"Xenon", b"Zanzibar"],                     # start bytes Q, X, Z
    "bytes_m1": lambda: [b"Quartz", b"Quebec", b"Zanzibar"],                    # start bytes Q, Z
}
# haystack alphabet per set: the byte-set scan retires when its needles are in more than one offset
# out of 64, so its haystacks are lower-case text in which Q, X, Z only occur where planted
HAY_ALPHABET = {"bytes_m0": (0x61, 0x7A), "bytes_m1": (0x61, 0x7A)}

_pats_cache = {}


def patterns(name):
    if name not in _pats_cache:
        _pats_cache[name] = PATTERN_SETS[name]()
    return _pats_cache[name]


def make_hay(pset, nbytes, ci=False, seed=5):
    """Random text with one planted occurrence per ~4 KiB everywhere and one per ~128 bytes over two
    stretches (the start and the middle), so that the slot queues fill and drain."""
    pats = patterns(pset)
    hay = np.empty(nbytes, dtype=np.uint8)
    W.fill_haystack(hay, seed, alphabet=HAY_ALPHABET.get(pset, (0x20, 0x7E)))
    W.plant(hay, pats, seed + 1, period=4096, window=2048)
    for lo, hi in ((0, nbytes // 8), (nbytes // 2, nbytes // 2 + nbytes // 16)):
        W.plant(hay[lo:hi], pats, seed + 2, period=128, window=64)
    if ci:
        W.flip_case(hay, seed + 3)
    return hay


def new_handle(pset, kind, ci, engine=ab.Engine.Auto):
    return (ab.AhoCorasick.builder().match_kind(kind).ascii_case_insensitive(ci).kind(ab.AhoCorasickKind.DFA)
            .build(patterns(pset)).set_engine(engine))


def oracle(pset, kind, ci):
    return O.Oracle(patterns(pset), match_kind=kind, ascii_case_insensitive=ci, kind=O.KIND_DFA)


def is_masked(p):
    return p.fold != 0 or p.kmask != 0xFFFFFFFF


def variant_of(p):
    """The variant index of launch_prefilter: 0 stride 1, 1 stride 1 + dense, 2 stride 2 narrow, 3 wide."""
    if p.dense:
        return 1
    return (3 if p.wide else 2) if p.stride == 2 else 0


def dyn_of(flags):
    """The tile distribution enqueue_prefilter_range derives from the experiment flags."""
    return 0 if flags & 32 else (2 if flags & 16 else 1)


VARIANT_NAME = {0: "stride1", 1: "stride1-dense", 2: "stride2-narrow", 3: "stride2-wide"}
TILES = {32: "static", 0: "percta", 16: "global"}
MODE_OF_API = {"overlapping": 0, "standard": 0, "leftmost": 1}

# ---- the instantiation matrix ------------------------------------------------------------------------
# (pattern set, match kind, case folding, API, expected (variant, masked)).  Every row runs under all
# three tile distributions.  MODE 0 rows alternate between find_overlapping_iter and Standard find_iter;
# MODE 1 rows between leftmost-first and leftmost-longest.
COMBOS = [
    ("k4_ap", 0, False, "overlapping", (0, False)),
    ("dense", 0, False, "standard", (1, False)),
    ("cfg2", 0, False, "overlapping", (2, False)),
    ("cfg4", 0, False, "standard", (3, False)),
    ("k3", 0, False, "standard", (0, True)),
    ("dense", 0, True, "overlapping", (1, True)),
    ("cfg2", 0, True, "standard", (2, True)),
    ("cfg4", 0, True, "overlapping", (3, True)),
    ("k4_ap", 2, False, "leftmost", (0, False)),
    ("dense", 1, False, "leftmost", (1, False)),
    ("cfg2", 1, False, "leftmost", (2, False)),
    ("cfg4", 2, False, "leftmost", (3, False)),
    ("k3", 1, False, "leftmost", (0, True)),
    ("dense", 2, True, "leftmost", (1, True)),
    ("cfg2", 1, True, "leftmost", (2, True)),
    ("cfg4", 1, True, "leftmost", (3, True)),
]
# the paths beside the fingerprint kernels, in both modes
EXTRA = [
    ("bytes_m0", 0, False, "overlapping", "bytescan"),
    ("bytes_m1", 1, False, "leftmost", "bytescan"),
    ("brute", 0, False, "overlapping", "brute"),
    ("brute", 1, False, "leftmost", "brute"),
]


def combo_id(c):
    pset, kind, ci, api, (variant, masked) = c
    return "m%d-%s-%s-%s-%s%s" % (MODE_OF_API[api], api, VARIANT_NAME[variant], "masked" if masked else "unmasked",
                                  pset, "-ci" if ci else "")


CASES = [(c, flags) for c in COMBOS for flags in (32, 0, 16)]
NARROW_BYTES = scaled(48 * MiB)   # per-CTA counter: every warp draws several tiles; global: > 1 super-tile round
SPAN = (4099, NARROW_BYTES - 777)  # unaligned start and end


def needed_answers(pset, kind, ci, api):
    """(name, function of the haystack) of every oracle answer a row compares with."""
    o = oracle(pset, kind, ci)
    out = []
    if api == "overlapping":
        # the overlapping stream over a span is the whole stream's matches inside the span
        out.append(("full", o.find_overlapping_iter_np))
    else:
        out.append(("full", o.find_iter_np))
        out.append(("span", lambda h: o.find_iter_np(h, span=SPAN)))
    if MODE_OF_API[api] == 0:
        out.append(("count", o.scan_overlapping_count))
    return out


@pytest.fixture(scope="module")
def matrix_inputs():
    """Haystacks (host + device) and oracle answers of every matrix row, computed once and shared by
    the three tile distributions; the oracle runs on a thread pool (it releases the GIL)."""
    hays, jobs = {}, []
    for pset, kind, ci, api, _ in COMBOS + [e[:4] + (None,) for e in EXTRA]:
        if (pset, ci) not in hays:
            h = make_hay(pset, NARROW_BYTES, ci)
            hays[(pset, ci)] = (h, to_device(torch.from_numpy(h)))
        for name, fn in needed_answers(pset, kind, ci, api):
            jobs.append(((pset, kind, ci, api, name), fn, hays[(pset, ci)][0]))
    with ThreadPoolExecutor(min(16, os.cpu_count() or 4)) as ex:
        futs = {key: ex.submit(fn, h) for key, fn, h in jobs}
        answers = {key: f.result() for key, f in futs.items()}
    return hays, answers


_handles = {}


def matrix_handle(pset, kind, ci):
    key = (pset, kind, ci)
    if key not in _handles:
        _handles[key] = new_handle(pset, kind, ci)
    return _handles[key]


def run_row(ac, api, ptr, n, span=None):
    if api == "overlapping":
        return ac.find_overlapping_iter_dev_np(ptr, n, span=span)[0]
    return ac.find_iter_dev_np(ptr, n, span=span)[0]


def check_row(pset, kind, ci, api, ac, inputs):
    hays, answers = inputs
    h, d = hays[(pset, ci)]
    n = h.size
    key = (pset, kind, ci, api)
    want = answers[key + ("full",)]
    assert len(want) > 1000
    got = run_row(ac, api, d.data_ptr(), n)
    assert ac.last_stats()["engine"] == PREFILTER
    assert_np_equal(got, want, key)
    s, e = SPAN
    sub = run_row(ac, api, d.data_ptr(), n, span=SPAN)
    if api == "overlapping":
        want_sub = want[(want["start"] >= s) & (want["end"] <= e)]
    else:
        want_sub = answers[key + ("span",)]
    assert_np_equal(sub, want_sub, key + ("span",))
    if MODE_OF_API[api] == 0:
        cnt, fnv, _ = ac.count_overlapping_dev(d.data_ptr(), n)
        assert ac.last_stats()["engine"] == PREFILTER
        assert (cnt, fnv) == answers[key + ("count",)], key


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("combo,flags", CASES, ids=["%s-%s" % (combo_id(c), TILES[f]) for c, f in CASES])
def test_instantiation(combo, flags, matrix_inputs):
    pset, kind, ci, api, (variant, masked) = combo
    ac = set_experiment(matrix_handle(pset, kind, ci), flags)
    p = plan_of(ac)
    assert p.supported and not p.brute and p.bs_n == 0
    assert (variant_of(p), is_masked(p)) == (variant, masked), (p.stride, p.wide, p.dense, p.fold, p.kmask)
    check_row(pset, kind, ci, api, ac, matrix_inputs)


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("row", EXTRA, ids=["m%d-%s-%s" % (MODE_OF_API[e[3]], e[4], e[3]) for e in EXTRA])
def test_bytescan_and_brute_paths(row, matrix_inputs):
    pset, kind, ci, api, path = row
    ac = new_handle(pset, kind, ci)   # a fresh handle: the byte-set scan has not been retired
    p = plan_of(ac)
    assert p.supported
    assert (p.bs_n > 0, bool(p.brute)) == (path == "bytescan", path == "brute")
    check_row(pset, kind, ci, api, ac, matrix_inputs)
    if path == "bytescan":
        assert plan_of(ac).bs_n > 0   # still the byte-set scan: its needles stayed rare
        assert 0 < ac.last_stats()["candidates"] < NARROW_BYTES // 64
    else:
        assert ac.last_stats()["candidates"] >= SPAN[1] - SPAN[0] - 64   # every position verified


def test_case_table_covers_every_instantiation():
    """Without a GPU: the plan of every matrix row (host-only build) maps to the launch_prefilter table
    index it claims, and together the rows reach all 48 kernel instantiations, the byte-set scan in both
    modes and the brute-force path in both modes."""
    reached = set()
    for (pset, kind, ci, api, (variant, masked)), flags in CASES:
        ac = (ab.AhoCorasick.builder().host_only(True).match_kind(kind).ascii_case_insensitive(ci)
              .kind(ab.AhoCorasickKind.DFA).build(patterns(pset)))
        p = plan_of(set_experiment(ac, flags))
        assert p.supported and not p.brute and p.bs_n == 0, (pset, kind, ci)
        assert (variant_of(p), is_masked(p)) == (variant, masked), (pset, kind, ci)
        reached.add((MODE_OF_API[api], int(is_masked(p)), dyn_of(flags), variant_of(p)))
    for pset, kind, ci, api, path in EXTRA:
        p = plan_of(ab.AhoCorasick.builder().host_only(True).match_kind(kind).ascii_case_insensitive(ci)
                    .kind(ab.AhoCorasickKind.DFA).build(patterns(pset)))
        if path == "bytescan":
            assert p.bs_n > 0
        else:
            assert p.brute and p.bs_n == 0
        reached.add((path, MODE_OF_API[api]))
    required = {(m, k, dyn, v) for m in (0, 1) for k in (0, 1) for dyn in (0, 1, 2) for v in range(4)}
    required |= {(path, m) for path in ("bytescan", "brute") for m in (0, 1)}
    assert required - reached == set()
    assert len(required) == 52


# ---- the global super-tile distribution over many rounds ---------------------------------------------
def sm_count():
    if ON_GPU:
        return torch.cuda.get_device_properties(0).multi_processor_count
    return int(os.environ.get("ACB_EMU_SMS", "3"))


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("pset,wide", [("cfg4", True), ("dense", False)], ids=["stride2-wide", "stride1-dense"])
def test_global_super_tiles_over_many_rounds(pset, wide):
    """Global super-tiles (256 tiles per CTA) with every CTA installing several: 512 MiB.  CTAs per SM
    from launch_prefilter's shared-memory formula (narrow: one 1 024-thread CTA, 227 088 B; wide: two
    512-thread CTAs), not measured.  Checked against the default tile distribution tuple for tuple, the
    walk engine (tuples, count + FNV) and the oracle on three 8 MiB windows."""
    n = scaled(512 * MiB)
    tile, per_sm = (2048, 2) if wide else (1024, 1)
    rounds = n / (sm_count() * per_sm * 256 * tile)
    assert rounds > 2, rounds
    pats = patterns(pset)
    d = torch.empty(n, dtype=torch.uint8, device="cuda" if ON_GPU else "cpu")
    W.torch_fill_config("cfg2", d, pats)
    ac = set_experiment(new_handle(pset, 0, False), 16)
    p = plan_of(ac)
    assert (variant_of(p), is_masked(p)) == ((3 if wide else 1), False)
    full, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n)
    assert ac.last_stats()["engine"] == PREFILTER
    cnt, fnv, _ = ac.count_overlapping_dev(d.data_ptr(), n)
    assert cnt == len(full) and cnt > n // 8192
    set_experiment(ac, 0)
    assert_np_equal(ac.find_overlapping_iter_dev_np(d.data_ptr(), n)[0], full, "per-CTA counter")
    walk = new_handle(pset, 0, False, engine=ab.Engine.Walk)
    assert_np_equal(walk.find_overlapping_iter_dev_np(d.data_ptr(), n)[0], full, "walk")
    assert walk.count_overlapping_dev(d.data_ptr(), n)[:2] == (cnt, fnv)
    assert walk.last_stats()["engine"] == int(ab.Engine.Walk)
    o = O.Oracle(pats, kind=O.KIND_DFA)
    win = min(8 * MiB, n // 4)
    for off in (0, n // 2 + 4096 * 7 + 3, n - win):
        w = d[off: off + win].cpu().numpy()
        want = o.find_overlapping_iter_np(w)
        got = full[(full["start"] >= off) & (full["end"] <= off + win)]
        assert len(got) == len(want)
        assert np.array_equal(got["pid"], want["pid"]) and np.array_equal(got["start"] - off, want["start"]) \
            and np.array_equal(got["end"] - off, want["end"])


# ---- guard bytes and alignments on device memory -----------------------------------------------------
GUARD_ENGINES = {   # name: (pattern set, match kind, expected path)
    "stride1": ("k3", 0, "fingerprint"),
    "stride2-narrow": ("cfg2", 0, "fingerprint"),
    "stride2-wide": ("cfg4", 0, "fingerprint"),
    "stride1-dense": ("dense", 0, "fingerprint"),
    "bytescan": ("bytes_m0", 0, "bytescan"),
    "brute": ("brute", 0, "brute"),
}
CUTS = (0, 1, 2, 3, 15, 16, 17, 20, 21, 33)


def _expect_path(ac, path):
    p = plan_of(ac)
    assert (p.bs_n > 0, bool(p.brute)) == (path == "bytescan", path == "brute")


def _put(buf, at, b):
    buf[at: at + len(b)] = np.frombuffer(b, dtype=np.uint8)


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("name", list(GUARD_ENGINES))
def test_guard_bytes_at_every_pointer_phase(name):
    """The haystack at 18 pointer phases inside a larger device buffer, its end and the span's end cut
    at 10 distances.  The bytes just past hay_len, just before span_start and just past span_end each
    complete an occurrence, so a kernel that reads or accepts a byte it does not own reports a match
    the oracle does not."""
    pset, kind, path = GUARD_ENGINES[name]
    pats = patterns(pset)
    p_end, p_mid = max(pats, key=len), sorted(pats, key=len)[len(pats) // 2]
    ac = new_handle(pset, kind, False)
    _expect_path(ac, path)
    o = oracle(pset, kind, False)
    base = make_hay(pset, 40 << 10, seed=9)
    W.plant(base, pats, 8, period=64, window=32)
    host = np.zeros(base.size + 64, dtype=np.uint8)
    dev = to_device(torch.from_numpy(host.copy()))
    for phase in range(18):
        for cut in CUTS:
            n = base.size - 24 - cut
            s = 4096 + 17 * phase + 1                    # one byte into an occurrence
            e = n - 21 - cut                             # an occurrence ends one byte past the span
            host[:] = 0
            view = host[phase: phase + base.size]
            view[:] = base
            _put(view, s - 1, p_mid)
            _put(view, e - (len(p_end) - 1), p_end)
            _put(view, n - (len(p_end) - 1), p_end)      # the haystack ends in p[:-1], byte n is p[-1]
            dev.copy_(torch.from_numpy(host))
            ptr = dev.data_ptr() + phase
            hay = view[:n]
            for span in ((0, n), (s, e)):
                got, _ = ac.find_overlapping_iter_dev_np(ptr, n, span=span)
                assert_np_equal(got, o.find_overlapping_iter_np(hay, span=span), (name, phase, cut, span))
                assert ac.last_stats()["engine"] == PREFILTER
    _expect_path(ac, path)


RAGGED = list(range(0, 70)) + [127, 128, 129, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096, 4097, 33000]


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("name", list(GUARD_ENGINES))
def test_ragged_sizes_on_every_engine(name):
    """The sizes of test_exact_size_device_buffers on the device, each followed by a guard byte that
    completes the occurrence the haystack ends with, on the Auto, Walk and Sequential engines."""
    pset, kind, path = GUARD_ENGINES[name]
    pats = patterns(pset)
    o = oracle(pset, kind, False)
    auto, walk, seq = (new_handle(pset, kind, False, engine=e)
                       for e in (ab.Engine.Auto, ab.Engine.Walk, ab.Engine.Sequential))
    rng = np.random.default_rng(17)
    alpha = np.array(range(*HAY_ALPHABET.get(pset, (0x20, 0x7E))), dtype=np.uint8)
    host = np.zeros(RAGGED[-1] + 64, dtype=np.uint8)
    dev = to_device(torch.from_numpy(host.copy()))
    for size in RAGGED:
        host[:] = alpha[rng.integers(0, alpha.size, size=host.size)]
        p = pats[size % len(pats)]
        if len(p) <= size + 1:
            _put(host, size + 1 - len(p), p)            # ends in p[:-1]; the byte past the haystack is p[-1]
        dev.copy_(torch.from_numpy(host))
        hay = host[:size].copy()
        ptr = dev.data_ptr() if size else 0
        want_ovl, want_it = o.find_overlapping_iter_np(hay), o.find_iter_np(hay)
        assert_np_equal(auto.find_overlapping_iter_dev_np(ptr, size)[0], want_ovl, (name, size))
        assert_np_equal(auto.find_iter_dev_np(ptr, size)[0], want_it, (name, size, "find_iter"))
        assert_np_equal(walk.find_overlapping_iter_dev_np(ptr, size)[0], want_ovl, (name, size, "walk"))
        assert_np_equal(seq.find_iter_dev_np(ptr, size)[0], want_it, (name, size, "sequential"))
    assert walk.last_stats()["engine"] == int(ab.Engine.Walk)
    assert seq.last_stats()["engine"] == int(ab.Engine.Sequential)
    _expect_path(auto, path)


# ---- host-copy paths ---------------------------------------------------------------------------------
HOST_HANDLES = {   # name: (pattern set, match kind)
    "stride2-m0": ("cfg2", 0),
    "stride2-m1": ("cfg2", 1),
    "bytescan-m0": ("bytes_m0", 0),
}
ODD_START = 1048577
# (span start, span length): below the 8 MiB staging threshold, at it, a ring sized to the span, one
# whole 64 MiB chunk, one chunk + 1 byte, three chunks from an odd start
HOST_SPANS = [(0, scaled(8 * MiB) - 1), (0, scaled(8 * MiB)), (0, scaled(40 * MiB)), (0, scaled(64 * MiB)),
              (0, scaled(64 * MiB) + 1), (ODD_START, scaled(130 * MiB) + 12345)]
SMALL_CHUNK = scaled(4 * MiB)
DEFAULT_CHUNK = 64 * MiB


def set_pipeline_chunk(ac, nbytes):
    ab._lib.acg_debug_set_pipeline_chunk.argtypes = [ctypes.c_void_p, ctypes.c_uint64]
    assert ab._lib.acg_debug_set_pipeline_chunk(ac._h, nbytes) == 0
    return ac


def host_hay(pset):
    n = ODD_START + HOST_SPANS[-1][1] + 4096
    hay = make_hay(pset, n, seed=21)
    pats = patterns(pset)
    # an occurrence across every chunk boundary counted from each span start (small and default chunks)
    for start in (0, ODD_START):
        k = 1
        while start + k * SMALL_CHUNK + 32 < n:
            p = pats[k % len(pats)]
            _put(hay, start + k * SMALL_CHUNK - len(p) // 2, p)
            k += 1
    return hay


@pytest.fixture(scope="module")
def host_inputs():
    """Per handle: the host haystack, its device copy and the oracle's answers for the spans up to 64 MiB."""
    out, hays, jobs = {}, {}, []
    for name, (pset, kind) in HOST_HANDLES.items():
        if pset not in hays:
            h = host_hay(pset)
            hays[pset] = (h, to_device(torch.from_numpy(h)))
        h, d = hays[pset]
        out[name] = {"hay": h, "dev": d}
        o = oracle(pset, kind, False)
        fn = o.find_overlapping_iter_np if kind == 0 else o.find_iter_np
        for s, ln in HOST_SPANS:
            if ln <= scaled(64 * MiB):
                jobs.append(((name, s, ln), fn, h, (s, s + ln)))
    with ThreadPoolExecutor(min(16, os.cpu_count() or 4)) as ex:
        futs = {key: ex.submit(fn, h, span) for key, fn, h, span in jobs}
        answers = {key: f.result() for key, f in futs.items()}
    return out, answers


def _host_search(ac, kind, hay, span):
    return ac.try_find_overlapping_iter_np(hay, span) if kind == 0 else ac.try_find_iter_np(hay, span)


def _dev_search(ac, kind, d, n, span):
    return (ac.find_overlapping_iter_dev_np if kind == 0 else ac.find_iter_dev_np)(d.data_ptr(), n, span=span)[0]


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("name", list(HOST_HANDLES))
def test_host_copy_paths(name, memory, host_inputs):
    """try_find_*_np from pageable (staged through the copy pool from 8 MiB on) and page-locked host
    memory, with the default 64 MiB pipeline chunk and with 4 MiB chunks: equal to the device-resident
    search of the same bytes, and to the oracle for the spans up to 64 MiB."""
    if memory == "pinned" and not ON_GPU:
        pytest.skip("page-locked memory needs a CUDA device")
    inputs, answers = host_inputs
    pset, kind = HOST_HANDLES[name]
    h, d = inputs[name]["hay"], inputs[name]["dev"]
    if memory == "pinned":
        t = torch.empty(h.size, dtype=torch.uint8, pin_memory=True)
        t.numpy()[:] = h
        src = t.numpy()
    else:
        src = h
    ac = new_handle(pset, kind, False)
    small = set_pipeline_chunk(new_handle(pset, kind, False), SMALL_CHUNK)
    for s, ln in HOST_SPANS:
        span = (s, s + ln)
        want = _dev_search(ac, kind, d, h.size, span)
        if (name, s, ln) in answers:
            assert_np_equal(want, answers[(name, s, ln)], (name, span, "device vs oracle"))
        assert_np_equal(_host_search(ac, kind, src, span), want, (name, memory, span))
        assert ac.last_stats()["engine"] == PREFILTER
        if ln > 2 * SMALL_CHUNK:
            assert_np_equal(_host_search(small, kind, src, span), want, (name, memory, span, "small chunks"))
    assert len(want) > HOST_SPANS[-1][1] // 4096 // 2
    if pset.startswith("bytes"):
        assert plan_of(ac).bs_n > 0 and plan_of(small).bs_n > 0


# ---- concurrency on the device -----------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_concurrent_searches_on_shared_handles():
    """8 threads on one handle (more than its 4 workspaces, so leases wait) mixing the device-resident,
    page-locked, pageable (staged through the shared copy pool), count and try_find entry points; at the
    same time a second handle's pageable searches and a byte-set-scan handle whose first concurrent
    searches retire the scan.  Every result is its precomputed answer and last_stats() is the caller's."""
    n = scaled(16 * MiB)   # on the device: above the 8 MiB staging threshold
    a_pats = patterns("cfg2")
    hay_a = make_hay("cfg2", n, seed=31)
    dev_a = to_device(torch.from_numpy(hay_a))
    pin_a = None
    if ON_GPU:
        t = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        t.numpy()[:] = hay_a
        pin_a = t.numpy()
    hay_b = make_hay("cfg2", n, seed=41)
    hay_c = np.frombuffer(b"aaaaab" * (max(scaled(4 * MiB), 128 << 10) // 6), dtype=np.uint8).copy()  # >= 64 KiB: may retire
    dev_c = to_device(torch.from_numpy(hay_c))
    a = new_handle("cfg2", 0, False)
    b = new_handle("cfg2", 1, False)
    c = ab.AhoCorasick.builder().kind(ab.AhoCorasickKind.DFA).build([b"aaab", b"aab"])
    assert plan_of(c).bs_n == 1
    oa = O.Oracle(a_pats, kind=O.KIND_DFA)
    with ThreadPoolExecutor(4) as ex:
        f_ovl = ex.submit(oa.find_overlapping_iter_np, hay_a)
        f_std = ex.submit(oa.find_iter_np, hay_a)
        f_b = ex.submit(O.Oracle(a_pats, match_kind=1, kind=O.KIND_DFA).find_iter_np, hay_b)
        f_c = ex.submit(O.Oracle([b"aaab", b"aab"], kind=O.KIND_DFA).find_overlapping_iter_np, hay_c)
        f_cnt = ex.submit(oa.scan_overlapping_count, hay_a)
        want_ovl, want_std, want_b, want_c, want_cnt = (f.result() for f in (f_ovl, f_std, f_b, f_c, f_cnt))
    span_f = (n // 3 + 1, n - 5)
    want_find = oa.try_find(hay_a, span_f)

    ops_a = {
        "dev_ovl": lambda: a.find_overlapping_iter_dev_np(dev_a.data_ptr(), n)[0],
        "dev_std": lambda: a.find_iter_dev_np(dev_a.data_ptr(), n)[0],
        "pageable": lambda: a.try_find_overlapping_iter_np(hay_a),
        "count": lambda: a.count_overlapping_dev(dev_a.data_ptr(), n)[:2],
        "find": lambda: (lambda m: m.as_tuple() if m else None)(a.try_find(hay_a, span_f)),
    }
    if pin_a is not None:
        ops_a["pinned"] = lambda: a.try_find_overlapping_iter_np(pin_a)
    expect = {"dev_ovl": want_ovl, "dev_std": want_std, "pageable": want_ovl, "pinned": want_ovl,
              "count": want_cnt, "find": want_find}
    # each entry point once, alone: the answer and the caller's raw match count
    raw_a = {}
    for k, fn in ops_a.items():
        got = fn()
        if isinstance(expect[k], np.ndarray):
            assert_np_equal(got, expect[k], k)
        else:
            assert got == expect[k], k
        raw_a[k] = a.last_stats()["raw_matches"]
    assert raw_a["dev_ovl"] == len(want_ovl)
    assert_np_equal(b.try_find_iter_np(hay_b), want_b, "b")
    raw_b = b.last_stats()["raw_matches"]

    errors, lock = [], threading.Lock()

    def check(tag, got, want, raw, want_raw):
        try:
            if isinstance(want, np.ndarray):
                assert_np_equal(got, want, tag)
            else:
                assert got == want, tag
            assert raw == want_raw, (tag, raw, want_raw)
        except AssertionError as e:
            with lock:
                errors.append(e)

    names = list(ops_a)

    def worker_a(i):
        for j in range(2 * len(names)):
            k = names[(i + j) % len(names)]
            got = ops_a[k]()
            check(("a", i, k), got, expect[k], a.last_stats()["raw_matches"], raw_a[k])

    def worker_b(i):
        for j in range(4):
            got = b.try_find_iter_np(hay_b)
            check(("b", i, j), got, want_b, b.last_stats()["raw_matches"], raw_b)

    def worker_c(i):
        for j in range(4):
            got = (c.find_overlapping_iter_dev_np(dev_c.data_ptr(), hay_c.size)[0] if (i + j) % 2
                   else c.try_find_overlapping_iter_np(hay_c))
            check(("c", i, j), got, want_c, c.last_stats()["raw_matches"], len(want_c))

    with ThreadPoolExecutor(12) as ex:
        futs = [ex.submit(worker_a, i) for i in range(8)] + [ex.submit(worker_b, i) for i in range(2)] + \
               [ex.submit(worker_c, i) for i in range(2)]
        for f in futs:
            f.result()
    assert not errors, errors[:3]
    assert plan_of(c).bs_n == 0   # the needles are everywhere: the scan retired during the concurrent searches
