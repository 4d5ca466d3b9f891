"""GPU parity tests: every search goes through the C ABI (libacb200.so) into the CUDA kernels and
is compared tuple-for-tuple (order included) with the CPU oracle / the committed golden vectors."""
import random

import numpy as np
import pytest

import aho_corasick_b200 as ab
import golden_util as G
import oracle_py as O
from aho_corasick_b200 import workload as W
from test_prefilter_plan import set_experiment

pytestmark = pytest.mark.gpu


def to_device(t):
    """The tensor on the GPU -- or unchanged under the CPU dry run of tests/emu (ACB_EMULATE=1),
    where "device" pointers are host pointers."""
    import torch
    return t.cuda() if torch.cuda.is_available() else t


AC = G.load("ac_vectors.json")
PK = G.load("packed_vectors.json")


def build(pats, match_kind=0, engine=ab.Engine.Auto, **kw):
    b = ab.AhoCorasick.builder().match_kind(match_kind)
    for k, v in kw.items():
        getattr(b, k)(v)
    return b.build(pats).set_engine(engine)


# Auto picks the prefilter engine whenever the automaton allows it; the second entry forces the
# state-transition walk (overlapping) / the single-lane reference loop (find_iter).
OVERLAPPING_ENGINES = [ab.Engine.Auto, ab.Engine.Walk]
FIND_ITER_ENGINES = [ab.Engine.Auto, ab.Engine.Sequential]


def tuples(ms):
    return [m.as_tuple() for m in ms]


def np_tuples(r):
    return list(zip(r["pid"].tolist(), r["start"].tolist(), r["end"].tolist()))


def assert_np_equal(got, want, ctx=None):
    assert len(got) == len(want), (len(got), len(want), ctx)
    for k in ("pid", "start", "end"):
        if not np.array_equal(got[k], want[k]):
            i = int(np.nonzero(got[k] != want[k])[0][0])
            raise AssertionError((k, i, np_tuples(got[max(0, i - 2): i + 3]), np_tuples(want[max(0, i - 2): i + 3]), ctx))


# ---- golden vectors through the device path (DFA rows of src/tests.rs:808-860, 937-994) -------
@pytest.mark.parametrize("engine", FIND_ITER_ENGINES)
@pytest.mark.parametrize("combo", list(G.COMBO_DFA) + ["default"])
@pytest.mark.parametrize("coll,kind", G.NON_OVERLAPPING_COLLECTIONS)
def test_golden_find_iter(coll, kind, combo, engine):
    kw = {k: v for k, v in G.COMBO[combo].items()}
    for t in G.collection(AC, coll):
        ac = build(t["patterns"], kind, engine=engine, **kw)
        assert tuples(ac.find_iter(t["haystack"])) == t["matches"], (t["name"], combo)


@pytest.mark.parametrize("engine", OVERLAPPING_ENGINES)
@pytest.mark.parametrize("combo", list(G.COMBO_DFA) + ["default"])
def test_golden_find_overlapping_iter(combo, engine):
    kw = {k: v for k, v in G.COMBO[combo].items()}
    for t in G.collection(AC, "AC_STANDARD_OVERLAPPING"):
        ac = build(t["patterns"], 0, engine=engine, **kw)
        assert tuples(ac.find_overlapping_iter(t["haystack"])) == t["matches"], (t["name"], combo)


@pytest.mark.parametrize("combo", ["dfa_default", "dfa_start_both"])
@pytest.mark.parametrize("coll,kind", G.ANCHORED)
def test_golden_anchored(coll, kind, combo):
    kw = dict(G.ANCHORED_COMBO[combo])
    for t in G.collection(AC, coll):
        ac = build(t["patterns"], kind, **kw)
        assert tuples(ac.find_iter(t["haystack"], anchored=ab.Anchored.Yes)) == t["matches"], (t["name"], combo)


def test_golden_ascii_case_insensitive():
    for kind, groups, overlapping in [
        (0, ["ASCII_CASE_INSENSITIVE", "ASCII_CASE_INSENSITIVE_NON_OVERLAPPING"], False),
        (0, ["ASCII_CASE_INSENSITIVE", "ASCII_CASE_INSENSITIVE_OVERLAPPING"], True),
        (1, ["ASCII_CASE_INSENSITIVE", "ASCII_CASE_INSENSITIVE_NON_OVERLAPPING"], False),
        (2, ["ASCII_CASE_INSENSITIVE", "ASCII_CASE_INSENSITIVE_NON_OVERLAPPING"], False),
    ]:
        for g in groups:
            for t in AC["groups"][g]:
                ac = build(t["patterns"], kind, ascii_case_insensitive=True, kind=ab.AhoCorasickKind.DFA)
                got = ac.find_overlapping_iter(t["haystack"]) if overlapping else ac.find_iter(t["haystack"])
                assert tuples(got) == t["matches"], (t["name"], kind, overlapping)


def test_readme_and_doc_examples():
    hay = b"Nobody likes maple in their apple flavored Snapple."
    assert tuples(ab.AhoCorasick.new([b"apple", b"maple", b"Snapple"]).find_iter(hay)) == \
        [(1, 13, 18), (0, 28, 33), (2, 43, 50)]
    pats, hay = [b"append", b"appendage", b"app"], b"append the app to the appendage"
    assert tuples(build(pats).find_overlapping_iter(hay)) == \
        [(2, 0, 3), (0, 0, 6), (2, 11, 14), (2, 22, 25), (0, 22, 28), (1, 22, 31)]
    assert tuples(build(pats, 1).find_iter(hay)) == [(0, 0, 6), (2, 11, 14), (0, 22, 28)]
    assert tuples(build(pats, 2).find_iter(hay)) == [(0, 0, 6), (2, 11, 14), (1, 22, 31)]
    ac = build(pats, 1)
    assert ac.find(hay).as_tuple() == (0, 0, 6)
    assert ac.is_match(hay) and not ac.is_match(b"xyz")
    assert ac.find(b"abc") is None


# ---- packed vectors with the 3 x 261 "Z" padding sweep (src/packed/tests.rs:42-92); on the device
# the padding doubles as a shard-alignment sweep --------------------------------------------------
@pytest.mark.parametrize("coll,kind", [("PACKED_LEFTMOST_FIRST", 1), ("PACKED_LEFTMOST_LONGEST", 2)])
def test_packed_vectors_padding_sweep(coll, kind):
    for t in G.collection(PK, coll):
        ac = build(t["patterns"], kind, kind=ab.AhoCorasickKind.DFA)
        for off in list(range(0, 40)) + [63, 64, 65, 127, 128, 129, 255, 256, 257, 260]:
            z = b"Z" * off
            sh = [(p, s + off, e + off) for p, s, e in t["matches"]]
            assert tuples(ac.find_iter(z + t["haystack"])) == sh, (t["name"], off, "prefix")
            assert tuples(ac.find_iter(t["haystack"] + z)) == list(t["matches"]), (t["name"], off, "suffix")
            assert tuples(ac.find_iter(z + t["haystack"] + z)) == sh, (t["name"], off, "both")


# ---- randomized differential tests vs the oracle ------------------------------------------------
def rand_case(rng, it, allow_empty):
    alphabet = [b"ab", b"abcd", bytes(range(256)), b"aAbBcC ", b"abcdefghijklmnopqrstuvwxyz"][it % 5]
    npat = rng.choice([1, 2, 5, 20, 200])
    lo = 0 if (allow_empty and it % 6 == 0) else 1
    pats = [bytes(rng.choice(alphabet) for _ in range(rng.randint(lo, rng.choice([3, 8, 20]))))
            for _ in range(npat)]
    if it % 4 == 0:
        pats += [pats[0], pats[-1][:2] or b"a"]
    n = rng.choice([0, 1, 7, 100, 1000, 5000, 70000, 300000])
    hay = np.frombuffer(bytes(rng.choice(alphabet) for _ in range(min(n, 5000))), dtype=np.uint8)
    if n > 5000:
        reps = (n + hay.size - 1) // hay.size
        hay = np.tile(hay, reps)[:n].copy()
        # break the periodicity a little
        idx = np.array([rng.randrange(n) for _ in range(50)])
        hay[idx] = np.frombuffer(bytes(rng.choice(alphabet) for _ in range(50)), dtype=np.uint8)
    s = rng.randint(0, hay.size)
    e = rng.randint(s, hay.size)
    span = (s, e) if it % 3 == 0 else None
    return pats, hay, span, alphabet == b"aAbBcC "


@pytest.mark.parametrize("engine", OVERLAPPING_ENGINES)
def test_random_overlapping_vs_oracle(engine):
    rng = random.Random(0x6A11)
    used = set()
    for it in range(120):
        pats, hay, span, ci = rand_case(rng, it, allow_empty=True)
        kw = {"ascii_case_insensitive": ci, "byte_classes": it % 7 != 0}
        ac = build(pats, 0, engine=engine, kind=ab.AhoCorasickKind.DFA, **kw)
        o = O.Oracle(pats, kind=O.KIND_DFA, **kw)
        assert_np_equal(ac.try_find_overlapping_iter_np(hay, span), o.find_overlapping_iter_np(hay, span),
                        (it, pats[:5], hay.size, span))
        used.add(ac.last_stats()["engine"])
    if engine == ab.Engine.Auto:
        assert int(ab.Engine.Prefilter) in used and int(ab.Engine.Walk) in used  # empty patterns -> walk
    else:
        assert used == {int(ab.Engine.Walk)}


@pytest.mark.parametrize("engine", FIND_ITER_ENGINES)
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_random_find_iter_vs_oracle(kind, engine):
    rng = random.Random(0xF17E + kind)
    used = set()
    for it in range(90):
        pats, hay, span, ci = rand_case(rng, it, allow_empty=True)
        if engine == ab.Engine.Sequential and hay.size > 70000:
            hay = hay[:70000].copy()
            span = None
        kw = {"ascii_case_insensitive": ci}
        ac = build(pats, kind, engine=engine, kind=ab.AhoCorasickKind.DFA, **kw)
        o = O.Oracle(pats, match_kind=kind, kind=O.KIND_DFA, prefilter=False, **kw)
        assert_np_equal(ac.try_find_iter_np(hay, span), o.find_iter_np(hay, span), (it, pats[:5], hay.size, span))
        used.add(ac.last_stats()["engine"])
    if engine == ab.Engine.Auto:
        assert int(ab.Engine.Prefilter) in used


def test_pathological_chains():
    """ab/ba on ababab...: per-start candidates all overlap, so the whole haystack is one run of
    the chain resolution (SURVEY.md section 7b) -- must still be exact."""
    hay = np.frombuffer(b"ab" * 20000 + b"xx" + b"ba" * 3000, dtype=np.uint8)
    for kind in (0, 1, 2):
        ac = build([b"ab", b"ba"], kind, kind=ab.AhoCorasickKind.DFA)
        o = O.Oracle([b"ab", b"ba"], match_kind=kind, kind=O.KIND_DFA)
        assert_np_equal(ac.try_find_iter_np(hay), o.find_iter_np(hay), kind)
        assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    pats = [b"aaaa", b"aa", b"a", b"aaaaaaa"]
    hay = np.frombuffer(b"a" * 30001, dtype=np.uint8)
    for kind in (0, 1, 2):
        ac = build(pats, kind, kind=ab.AhoCorasickKind.DFA)
        o = O.Oracle(pats, match_kind=kind, kind=O.KIND_DFA)
        assert_np_equal(ac.try_find_iter_np(hay), o.find_iter_np(hay), kind)
    ac = build(pats, 0, kind=ab.AhoCorasickKind.DFA)
    assert_np_equal(ac.try_find_overlapping_iter_np(hay), O.Oracle(pats, kind=O.KIND_DFA).find_overlapping_iter_np(hay))


def test_adopted_reference_tables():
    """acg_dfa_create: the tables come from elsewhere (here: the oracle's restatement of the
    reference builder) -- exactly what a Rust -sys shim would pass."""
    pats, hay, _ = W.make_config("cfg2", 4 << 20)
    o = O.Oracle(pats, kind=O.KIND_DFA)
    t = o.dfa()
    t["start_kind"] = 0
    ac = ab.AhoCorasick.from_dfa_tables(t)
    assert_np_equal(ac.try_find_overlapping_iter_np(hay), o.find_overlapping_iter_np(hay))


# ---- BASELINE config 2 at reduced size, full tuple stream; and a size-independent property ------
@pytest.mark.parametrize("cfg,kind,ci", [("cfg3", 1, True), ("cfg3", 2, True), ("cfg4", 1, False), ("cfg2", 0, False)])
def test_config3_4_reduced_find_iter_parity(cfg, kind, ci):
    """BASELINE configs 3 (case-insensitive LeftmostFirst non-overlapping) and 4 (50 literals,
    the pattern set for which the reference activates Fat Teddy) at 32 MiB, full tuple parity."""
    import torch
    pats = W.make_patterns(W.CONFIGS[cfg]["n_patterns"], W.CONFIGS[cfg]["pattern_seed"])
    t = torch.empty(32 << 20, dtype=torch.uint8)
    W.torch_fill_config(cfg, t, pats, chunk=1 << 24)
    hay = t.numpy()
    ac = build(pats, kind, ascii_case_insensitive=ci, kind=ab.AhoCorasickKind.DFA)
    o = O.Oracle(pats, match_kind=kind, ascii_case_insensitive=ci, kind=O.KIND_DFA)
    want = o.find_iter_np(hay)
    assert len(want) > 7000
    assert_np_equal(ac.try_find_iter_np(hay), want)
    assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    d = to_device(t)
    got, ms = ac.find_iter_dev_np(d.data_ptr(), hay.size)
    assert_np_equal(got, want)
    if cfg == "cfg4":
        assert ac.prefilter_kind() == 4 and o.prefilter_kind == O.PRE_PACKED  # packed (Teddy) in the reference
        assert ac.packed_variant() == {"fat": True, "mask_len": 4}


@pytest.mark.parametrize("engine", OVERLAPPING_ENGINES)
def test_config2_reduced_full_tuple_parity(engine):
    import torch
    pats, hay, planted = W.make_config("cfg2", 64 << 20)
    ac = build(pats, 0, engine=engine, kind=ab.AhoCorasickKind.DFA)
    o = O.Oracle(pats, kind=O.KIND_DFA)
    want = o.find_overlapping_iter_np(hay)
    assert len(want) >= planted
    d = to_device(torch.from_numpy(hay))
    got, ms = ac.find_overlapping_iter_dev_np(d.data_ptr(), hay.size)
    assert_np_equal(got, want)
    # host-buffer entry point (H2D inside the call) gives the same stream
    assert_np_equal(ac.try_find_overlapping_iter_np(hay), want)
    # count + FNV of the ordered stream agree with the oracle's scalar scan loop
    cnt, fnv, _ = ac.count_overlapping_dev(d.data_ptr(), hay.size)
    assert (cnt, fnv) == o.scan_overlapping_count(hay)
    # property: the stream over a span equals the full stream filtered to matches inside the span
    s, e = 12345677, 50000003
    sub, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), hay.size, span=(s, e))
    keep = (want["start"] >= s) & (want["end"] <= e)
    assert_np_equal(sub, want[keep])


def test_pipelined_host_path_multi_chunk():
    """Host haystacks larger than one 64 MiB staging chunk are copied and scanned chunk by chunk
    (copy and scan overlap); the stream must equal the one-shot device-resident scan."""
    import torch
    pats = W.make_patterns(5000, W.CONFIGS["cfg2"]["pattern_seed"])
    t = torch.empty(200 << 20, dtype=torch.uint8)
    W.torch_fill_config("cfg2", t, pats, chunk=1 << 24)
    hay = t.numpy()
    d = to_device(t)
    for kind, overlapping in ((0, True), (0, False), (1, False)):
        ac = build(pats, kind, kind=ab.AhoCorasickKind.DFA)
        if overlapping:
            want, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), hay.size)
            got = ac.try_find_overlapping_iter_np(hay)
            sub = ac.try_find_overlapping_iter_np(hay, span=(70 << 20 | 5, (190 << 20) + 3))
            keep = (want["start"] >= (70 << 20 | 5)) & (want["end"] <= (190 << 20) + 3)
            assert_np_equal(sub, want[keep])
        else:
            want, _ = ac.find_iter_dev_np(d.data_ptr(), hay.size)
            got = ac.try_find_iter_np(hay)
        assert len(want) > 40000
        assert_np_equal(got, want, (kind, overlapping))


def test_full_size_properties_config2():
    """BASELINE config 2 at its full size (4 GiB, device-generated).  The oracle cannot scan 4 GiB
    in test time, so parity is carried by size-independent properties: (1) the two independent
    engines (sharded state-transition walk vs. prefilter + verify) produce the same ordered stream
    (count + FNV of every tuple); (2) a checksum of checksums: the stream over the whole haystack
    equals the concatenation of the streams over two half spans plus the matches that straddle the
    cut; (3) every planted pattern is reported; (4) the oracle agrees on sampled 8 MiB windows."""
    import torch
    n = 4 << 30
    pats = W.make_patterns(5000, W.CONFIGS["cfg2"]["pattern_seed"])
    try:
        d = torch.empty(n, dtype=torch.uint8, device="cuda")
    except RuntimeError:
        pytest.skip("not enough device memory for the 4 GiB haystack")
    planted = W.torch_fill_config("cfg2", d, pats)
    ac = build(pats, 0, kind=ab.AhoCorasickKind.DFA)
    cnt_p, fnv_p, _ = ac.count_overlapping_dev(d.data_ptr(), n)
    assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    ac.set_engine(ab.Engine.Walk)
    cnt_w, fnv_w, _ = ac.count_overlapping_dev(d.data_ptr(), n)
    assert ac.last_stats()["engine"] == int(ab.Engine.Walk)
    assert (cnt_p, fnv_p) == (cnt_w, fnv_w)
    assert cnt_p >= planted
    ac.set_engine(ab.Engine.Auto)
    # global super-tiles (ACG_EXP_GLOBAL_TILES = 16): one chunk spans the whole 4 GiB region, so the
    # kernel's queued 32-bit offsets go through its 2 GiB windows
    set_experiment(ac, 16)
    assert ac.count_overlapping_dev(d.data_ptr(), n)[:2] == (cnt_p, fnv_p)
    assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    set_experiment(ac, 0)
    full, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n)
    assert len(full) == cnt_p
    cut = (2 << 30) + 12345
    left, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n, span=(0, cut))
    right, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n, span=(cut, n))
    straddle = full[(full["start"] < cut) & (full["end"] > cut)]
    assert len(left) + len(right) + len(straddle) == len(full)
    assert_np_equal(left, full[full["end"] <= cut])
    assert_np_equal(right, full[full["start"] >= cut])
    o = O.Oracle(pats, kind=O.KIND_DFA)
    for off in (0, (1 << 30) + 4096 * 7 + 3, n - (8 << 20)):
        w = d[off: off + (8 << 20)].cpu().numpy()
        want = o.find_overlapping_iter_np(w)
        got = full[(full["start"] >= off) & (full["end"] <= off + (8 << 20))]
        assert len(got) == len(want)
        assert np.array_equal(got["pid"], want["pid"]) and np.array_equal(got["start"] - off, want["start"]) \
            and np.array_equal(got["end"] - off, want["end"])


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("device_fill", [False, True])
def test_full_size_properties_config5(device_fill):
    """BASELINE config 5's automaton at its full 100 000 patterns (dense-set kernel variant, 414 MB
    table), host-built and device-built, on a 2 GiB device-generated haystack: the two independent
    engines agree on count + FNV of the whole ordered stream, whole = left + right + straddlers, and
    the oracle agrees tuple for tuple on sampled 8 MiB windows."""
    import torch
    n = 2 << 30
    c = W.CONFIGS["cfg5"]
    pats = W.make_patterns(c["n_patterns"], c["pattern_seed"])
    assert len(pats) == 100000
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    planted = W.torch_fill_config("cfg5", d, pats)
    b = ab.AhoCorasick.builder().kind(ab.AhoCorasickKind.DFA)
    if device_fill:
        b.device_fill(True)
    ac = b.build(pats)
    cnt_p, fnv_p, _ = ac.count_overlapping_dev(d.data_ptr(), n)
    assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    ac.set_engine(ab.Engine.Walk)
    cnt_w, fnv_w, _ = ac.count_overlapping_dev(d.data_ptr(), n)
    assert ac.last_stats()["engine"] == int(ab.Engine.Walk)
    assert (cnt_p, fnv_p) == (cnt_w, fnv_w)
    assert cnt_p >= planted
    ac.set_engine(ab.Engine.Auto)
    full, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n)
    assert len(full) == cnt_p
    cut = (1 << 30) + 54321
    left, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n, span=(0, cut))
    right, _ = ac.find_overlapping_iter_dev_np(d.data_ptr(), n, span=(cut, n))
    straddle = full[(full["start"] < cut) & (full["end"] > cut)]
    assert len(left) + len(right) + len(straddle) == len(full)
    assert_np_equal(left, full[full["end"] <= cut])
    assert_np_equal(right, full[full["start"] >= cut])
    o = O.Oracle(pats, kind=O.KIND_DFA)
    for off in (0, (1 << 30) + 4096 * 7 + 3, n - (8 << 20)):
        w = d[off: off + (8 << 20)].cpu().numpy()
        want = o.find_overlapping_iter_np(w)
        got = full[(full["start"] >= off) & (full["end"] <= off + (8 << 20))]
        assert len(got) == len(want)
        assert np.array_equal(got["pid"], want["pid"]) and np.array_equal(got["start"] - off, want["start"]) \
            and np.array_equal(got["end"] - off, want["end"])


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("cfg,kind,ci", [("cfg3", 1, True), ("cfg4", 1, False)])
def test_full_size_properties_config3_4(cfg, kind, ci):
    """BASELINE configs 3 and 4 at their full size (4 GiB, find_iter, leftmost-first).  Size-independent
    properties: the list is ordered and non-overlapping; every reported span holds its pattern's bytes
    (checked on the device for all ~10^6 matches); every planted occurrence lies inside a reported
    match or overlaps one; on sampled windows that begin at a reported match end (so that the
    iterator's cursor is the same) the list equals the oracle's and the single-lane restatement of
    the reference loop (seq_find_kernel, the second device engine) tuple for tuple."""
    import torch
    n = 4 << 30
    c = W.CONFIGS[cfg]
    pats = W.make_patterns(c["n_patterns"], c["pattern_seed"])
    try:
        d = torch.empty(n, dtype=torch.uint8, device="cuda")
    except RuntimeError:
        pytest.skip("not enough device memory for the 4 GiB haystack")
    planted = W.torch_fill_config(cfg, d, pats)
    ac = build(pats, kind, ascii_case_insensitive=ci, kind=ab.AhoCorasickKind.DFA)
    full, _ = ac.find_iter_dev_np(d.data_ptr(), n)
    assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    st, en, pid = full["start"].astype(np.int64), full["end"].astype(np.int64), full["pid"].astype(np.int64)
    assert len(full) >= planted * 0.98   # a planted occurrence can be shadowed by a match that overlaps it
    assert bool(np.all(st[1:] >= en[:-1])) and bool(np.all(en > st))
    # every span spells its pattern (ASCII case folded for cfg 3)
    lens = np.array([len(p) for p in pats], dtype=np.int64)
    assert np.array_equal(en - st, lens[pid])
    maxlen = int(lens.max())
    table = np.zeros((len(pats), maxlen), dtype=np.uint8)
    for i, p in enumerate(pats):
        table[i, :len(p)] = np.frombuffer(p, dtype=np.uint8)

    def fold(x):
        if not ci:
            return x
        up = (x >= 65) & (x <= 90)
        return torch.where(up, x + 32, x)
    t_table = torch.from_numpy(table).cuda()
    t_st, t_pid, t_len = torch.from_numpy(st).cuda(), torch.from_numpy(pid).cuda(), torch.from_numpy(en - st).cuda()
    ar = torch.arange(maxlen, device="cuda")
    for lo in range(0, len(full), 1 << 18):
        sl = slice(lo, lo + (1 << 18))
        mask = ar[None, :] < t_len[sl][:, None]
        idx = (t_st[sl][:, None] + ar[None, :]).clamp_(max=n - 1)
        hb = fold(d[idx])
        pb = fold(t_table[t_pid[sl]])
        assert bool(torch.all((hb == pb) | ~mask))
    # sampled windows, starting where the iterator's cursor is known
    o = O.Oracle(pats, match_kind=kind, ascii_case_insensitive=ci, kind=O.KIND_DFA)
    win = 4 << 20
    for off in (0, (1 << 30) + 4096 * 7 + 3, (3 << 30) + 999, n - win - 4096):
        i0 = int(np.searchsorted(en, off))
        ws = int(en[i0]) if off else 0
        we = min(n, ws + win)
        w = d[ws:we].cpu().numpy()
        want = o.find_iter_np(w)
        safe = we - ws - maxlen     # a match that starts before this offset is decided by bytes inside the window
        want = want[want["start"].astype(np.int64) < safe]
        got = full[(st >= ws) & (st < ws + safe)]
        assert len(got) == len(want) and len(want) > 500
        assert np.array_equal(got["pid"], want["pid"]) and np.array_equal(got["start"] - ws, want["start"]) \
            and np.array_equal(got["end"] - ws, want["end"])
        # second device engine on the same window
        ac.set_engine(ab.Engine.Sequential)
        seq, _ = ac.find_iter_dev_np(d.data_ptr(), n, span=(ws, we))
        assert ac.last_stats()["engine"] == int(ab.Engine.Sequential)
        ac.set_engine(ab.Engine.Auto)
        pf, _ = ac.find_iter_dev_np(d.data_ptr(), n, span=(ws, we))
        assert_np_equal(seq, pf, (cfg, off))
        keep = seq["start"].astype(np.int64) < ws + safe
        assert_np_equal(seq[keep], got, (cfg, off, "seq vs full"))


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_find_single_vs_oracle(kind):
    """AhoCorasick::try_find (src/ahocorasick.rs:1021): windowed device scan vs the oracle."""
    rng = random.Random(0xF1D0 + kind)
    for it in range(80):
        pats, hay, span, ci = rand_case(rng, it, allow_empty=(it % 5 == 0))
        kw = {"ascii_case_insensitive": ci}
        ac = build(pats, kind, kind=ab.AhoCorasickKind.DFA, **kw)
        # same (default) prefilter knob as the product: with the packed prefilter attached, the
        # reference's unanchored try_find returns the leftmost match even under `earliest`
        o = O.Oracle(pats, match_kind=kind, kind=O.KIND_DFA, **kw)
        for earliest in (False, True):
            got = ac.try_find(hay, span, earliest=earliest)
            want = o.try_find(hay, span, earliest=earliest)
            assert (got.as_tuple() if got else None) == want, (it, pats[:4], hay.size, span, earliest)
        assert ac.is_match(hay, span) == (o.try_find(hay, span, earliest=True) is not None)


def test_find_far_match_multi_window():
    """The first match sits behind several scan windows (1 MiB, 16 MiB, ...)."""
    hay = np.full(40 << 20, ord("x"), dtype=np.uint8)
    hay[(30 << 20) + 5: (30 << 20) + 11] = np.frombuffer(b"needle", dtype=np.uint8)
    hay[(1 << 20) - 2: (1 << 20) + 1] = np.frombuffer(b"nee", dtype=np.uint8)   # near miss on a window edge
    for kind in (0, 1, 2):
        ac = build([b"needle", b"need", b"zzz"], kind, kind=ab.AhoCorasickKind.DFA)
        o = O.Oracle([b"needle", b"need", b"zzz"], match_kind=kind, kind=O.KIND_DFA)
        assert ac.try_find(hay).as_tuple() == o.try_find(hay)
        assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
        assert ac.try_find(hay, span=(0, (30 << 20) + 8)) is None
        assert ac.is_match(hay) and not ac.is_match(hay[: 30 << 20])
    # Standard semantics across a window edge: the earliest END wins even if it starts later
    pats = [b"a" + b"b" * 15, b"bb"]
    hay = np.full(3 << 20, ord("x"), dtype=np.uint8)
    hay[(1 << 20) - 3: (1 << 20) + 13] = np.frombuffer(pats[0], dtype=np.uint8)
    ac = build(pats, 0, kind=ab.AhoCorasickKind.DFA)
    assert ac.try_find(hay).as_tuple() == O.Oracle(pats, kind=O.KIND_DFA).try_find(hay)


def _apply(hay: bytes, matches, reps):
    out, last = bytearray(), 0
    for pid, s, e in matches:
        out += hay[last:s] + reps[pid]
        last = e
    return bytes(out + hay[last:])


def test_replace_all_and_stream():
    """replace_all* / stream_find_iter are host glue over find_iter (SURVEY.md section 8f.3);
    examples from src/ahocorasick.rs:651-760 and the stream rows of src/tests.rs:999-1036."""
    import io
    pats = [b"append", b"appendage", b"app"]
    hay = b"append the app to the appendage"
    assert build(pats, 1).replace_all(hay.decode(), ["x", "y", "z"]) == "x the z to the xage"
    assert build(pats, 2).replace_all_bytes(hay, [b"x", b"y", b"z"]) == b"x the z to the y"
    ac = build(pats, 1)
    dst = bytearray()
    ac.replace_all_with(hay, dst, lambda m, txt, out: (out.extend(txt.upper()), m.pattern() != 2)[1])
    assert bytes(dst) == b"APPEND the APP to the appendage"   # stops after the first "app"
    with pytest.raises(ValueError):
        ac.replace_all_bytes(hay, [b"x"])
    # stream search == find_iter of the whole stream, for every Standard vector without empty patterns
    for t in G.collection(AC, "AC_STANDARD_NON_OVERLAPPING"):
        if any(len(p) == 0 for p in t["patterns"]):
            continue
        ac = build(t["patterns"], 0, kind=ab.AhoCorasickKind.DFA)
        for chunk in (1, 2, 3, 7, 64 << 20):
            got = [m.as_tuple() for m in ac.stream_find_iter(io.BytesIO(t["haystack"]), chunk_bytes=chunk)]
            assert got == t["matches"], (t["name"], chunk)
    # unsupported configurations, src/automaton.rs:1087-1103
    with pytest.raises(ab.MatchError) as e:
        list(build([b"a"], 1).stream_find_iter(io.BytesIO(b"a")))
    assert e.value.kind == "UnsupportedStream"
    with pytest.raises(ab.MatchError) as e:
        list(build([b"a", b""], 0).stream_find_iter(io.BytesIO(b"a")))
    assert e.value.kind == "UnsupportedEmpty"
    # a larger stream with matches that straddle block boundaries, against the oracle
    pats2 = W.make_patterns(200, 77)
    t = np.empty(3 << 20, dtype=np.uint8)
    W.fill_haystack(t, 99)
    W.plant(t, pats2, 5, period=512, window=256)
    o = O.Oracle(pats2, kind=O.KIND_DFA)
    ac = build(pats2, 0, kind=ab.AhoCorasickKind.DFA)
    want = o.find_iter(t)
    got = [m.as_tuple() for m in ac.stream_find_iter(io.BytesIO(t.tobytes()), chunk_bytes=(1 << 18) + 13)]
    assert got == want and len(want) > 5000
    out = io.BytesIO()
    reps = [b"<%d>" % i for i in range(len(pats2))]
    ac.try_stream_replace_all(io.BytesIO(t.tobytes()), out, reps, chunk_bytes=1 << 19)
    assert out.getvalue() == _apply(t.tobytes(), want, reps)


def test_dense_outputs_and_unselective_fingerprints():
    """Stress the slow paths: (1) far more matches than the initial tuple capacity (counter
    overflow -> regrow -> rescan), (2) pattern sets whose fingerprints cannot be selective (every
    byte starts a pattern: the kernel verifies every position), (3) steps with more first-probe
    hits than the compaction slots."""
    # (1) 3 matches per position on 2 MiB of 'a'  => ~6.3 M tuples
    pats = [b"a", b"aa", b"aaa"]
    hay = np.full(2 << 20, ord("a"), dtype=np.uint8)
    o = O.Oracle(pats, kind=O.KIND_DFA)
    for engine in OVERLAPPING_ENGINES:
        ac = build(pats, 0, engine=engine, kind=ab.AhoCorasickKind.DFA)
        got = ac.try_find_overlapping_iter_np(hay)
        assert len(got) == 3 * hay.size - 3
        assert_np_equal(got, o.find_overlapping_iter_np(hay), engine)
    for kind in (0, 1, 2):
        ac = build(pats, kind, kind=ab.AhoCorasickKind.DFA)
        assert_np_equal(ac.try_find_iter_np(hay), O.Oracle(pats, match_kind=kind, kind=O.KIND_DFA).find_iter_np(hay), kind)
    # (2) all 256 single bytes + a few longer patterns
    pats = [bytes([b]) for b in range(256)] + [b"abc", b"\x00\x01\x02\x03", b"zz"]
    rng = np.random.default_rng(5)
    hay = rng.integers(0, 256, size=300000, dtype=np.uint8)
    hay[1000:1003] = np.frombuffer(b"abc", dtype=np.uint8)
    ac = build(pats, 0, kind=ab.AhoCorasickKind.DFA)
    o = O.Oracle(pats, kind=O.KIND_DFA)
    assert_np_equal(ac.try_find_overlapping_iter_np(hay), o.find_overlapping_iter_np(hay))
    assert ac.last_stats()["engine"] == int(ab.Engine.Prefilter)
    assert ac.last_stats()["candidates"] >= hay.size - 64   # every position was verified
    for kind in (1, 2):
        ac = build(pats, kind, kind=ab.AhoCorasickKind.DFA)
        assert_np_equal(ac.try_find_iter_np(hay), O.Oracle(pats, match_kind=kind, kind=O.KIND_DFA).find_iter_np(hay))
    # (3) 4-byte fingerprints that hit at every position of a periodic haystack
    pats = [b"abababab", b"babababa", b"abab"]
    hay = np.frombuffer(b"ab" * 200000, dtype=np.uint8)
    ac = build(pats, 0, kind=ab.AhoCorasickKind.DFA)
    assert_np_equal(ac.try_find_overlapping_iter_np(hay), O.Oracle(pats, kind=O.KIND_DFA).find_overlapping_iter_np(hay))


def test_searches_accept_input_objects():
    """`Input` (src/util/search.rs:60-720) carries span / anchored / earliest into every search;
    the Teddy-prefilter range regression of src/tests.rs:1523-1530 written the reference's way."""
    ac = build([b"abcd", b"bcd", b"cd", b"b"], 1, start_kind=ab.StartKind.Both)
    hay = b"abcdabcd"
    assert tuples(ac.find_iter(ab.Input(hay))) == tuples(ac.find_iter(hay))
    assert tuples(ac.find_iter(ab.Input(hay).span((1, 8)))) == tuples(ac.find_iter(hay, span=(1, 8)))
    assert ac.find(ab.Input(hay).range(range(1, 8))).as_tuple() == ac.find(hay, span=(1, 8)).as_tuple()
    a = ac.find(ab.Input(hay).span((1, 8)).anchored(ab.Anchored.Yes))
    assert a.as_tuple() == ac.find(hay, span=(1, 8), anchored=ab.Anchored.Yes).as_tuple() == (1, 1, 4)
    assert ac.is_match(ab.Input(hay).span((5, 8)))
    assert not ac.is_match(ab.Input(hay).span((0, 1)))
    std = build([b"abcd", b"bcd", b"cd", b"b"], 0)
    assert tuples(std.find_overlapping_iter(ab.Input(hay).span((0, 4)))) == tuples(std.find_overlapping_iter(hay, span=(0, 4)))
    assert std.find(ab.Input(hay).earliest(True)).as_tuple() == std.find(hay, earliest=True).as_tuple()


def test_find_overlapping_with_state():
    """`find_overlapping` + `OverlappingState`, doc example of src/ahocorasick.rs:430-470."""
    ac = build([b"append", b"appendage", b"app"], 0)
    hay = b"append the app to the appendage"
    state = ab.OverlappingState.start()
    got = []
    while True:
        ac.find_overlapping(hay, state)
        m = state.get_match()
        if m is None:
            break
        got.append(m.as_tuple())
    assert got == [(2, 0, 3), (0, 0, 6), (2, 11, 14), (2, 22, 25), (0, 22, 28), (1, 22, 31)]
    with pytest.raises(ab.MatchError):
        build([b"a"], 1).try_find_overlapping(b"a", ab.OverlappingState.start())
