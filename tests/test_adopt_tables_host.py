"""CPU checks of acg_dfa_create (adopting a DFA built elsewhere, include/acb200.h): tables produced
by the oracle's restatement of the reference builder -- what a Rust -sys shim would pass -- are
accepted and reproduce the product builder's derived state; malformed descriptors are rejected
with ACG_E_INVALID_ARG instead of being indexed out of bounds later."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import aho_corasick_b200 as ab  # noqa: E402
import oracle_py as O  # noqa: E402
from aho_corasick_b200 import workload as W  # noqa: E402

SETS = [
    ([b"apple", b"maple", b"Snapple"], {}),
    ([b"append", b"appendage", b"app"], {"match_kind": 1}),
    ([b"", b"ab", b"b"], {}),
    ([], {}),
    ([b"Sam", b"Samwise", b"sam"], {"match_kind": 2, "ascii_case_insensitive": True}),
    ([b"abcd", b"bcd", b"cd", b"b"], {"match_kind": 1, "start_kind": 2}),
    (W.make_patterns(300, 9), {}),
]


def _adopt(t):
    return ab.AhoCorasick.from_dfa_tables(t)


@pytest.mark.parametrize("idx", range(len(SETS)))
def test_oracle_tables_are_adopted(idx):
    pats, kw = SETS[idx]
    o = O.Oracle(pats, kind=O.KIND_DFA, **kw)
    t = o.dfa()
    t["start_kind"] = kw.get("start_kind", 0)
    ac = _adopt(t)
    got = ac.tables()
    for k in ("trans", "byte_classes", "match_offsets", "match_pids", "pattern_lens"):
        assert np.array_equal(np.asarray(got[k]), np.asarray(t[k])[: len(got[k])]), k
    assert ac.patterns_len() == len(pats) and ac.match_kind() == kw.get("match_kind", 0)
    if ab.device_count() == 0:
        with pytest.raises(ab.DeviceError):   # adopted, but searches need the GPU
            ac.find_iter(b"xx")
    else:   # with a GPU the adopted automaton finds what the oracle finds
        hay = b"xx " + b" ".join(pats) + b" SAMWISE appendage xx"
        got, want = ac.try_find_iter_np(hay), o.find_iter_np(hay)
        assert len(got) == len(want)
        for k in ("pid", "start", "end"):
            assert np.array_equal(got[k], want[k]), k


def _valid():
    pats = [b"append", b"appendage", b"app", b"bar"]
    t = O.Oracle(pats, kind=O.KIND_DFA).dfa()
    t["start_kind"] = 0
    return {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in t.items()}


def _rejects(t):
    with pytest.raises(ab.DeviceError) as e:
        _adopt(t)
    assert e.value.code == -22


def test_malformed_descriptors_are_rejected():
    _adopt(_valid())
    t = _valid(); t["stride2"] = 9; _rejects(t)
    t = _valid(); t["alphabet_len"] = (1 << int(t["stride2"])) + 1; _rejects(t)
    t = _valid(); t["trans"] = t["trans"][:-1]; _rejects(t)                      # not a whole number of rows
    t = _valid(); t["trans"][5] = len(t["trans"]); _rejects(t)                   # next-state id out of range
    t = _valid(); t["trans"][5] = 3; _rejects(t)                                 # id not premultiplied
    t = _valid(); t["byte_classes"][65] = t["alphabet_len"]; _rejects(t)         # class beyond the alphabet
    t = _valid(); t["start_unanchored_id"] = len(t["trans"]); _rejects(t)
    t = _valid(); t["max_match_id"] = 0; _rejects(t)
    t = _valid(); t["match_pids"][0] = 99; _rejects(t)                           # pattern id beyond n_patterns
    t = _valid(); t["match_offsets"][1] = t["match_offsets"][-1] + 7; _rejects(t)  # non-monotone CSR
    t = _valid(); t["match_kind"] = 3; _rejects(t)
    t = _valid(); t["max_pattern_len"] = 2; _rejects(t)                          # a pattern longer than the maximum
    # the FAIL row (row 1, id == stride) is never a transition target or a start state: its id looks
    # like a match state to the kernels (non-zero, <= max_match_id) and would index match_offsets[-1]
    stride = 1 << int(_valid()["stride2"])
    t = _valid(); t["trans"][2 * stride + 1] = stride; _rejects(t)
    t = _valid(); t["start_unanchored_id"] = stride; _rejects(t)
    t = _valid(); t["start_anchored_id"] = stride; _rejects(t)


def test_builder_row_depth_equals_the_walked_depth_of_the_same_table():
    """The builder hands the trie depth of every row to the device engine (acb_build.hpp:
    HostDfa::row_depth); an adopted copy of the same table has it derived by a BFS over the
    transitions.  Both must agree row for row, for every match kind, with and without case folding,
    with 1-byte and duplicate patterns."""
    import random
    from test_prefilter_plan import plan_of
    rng = random.Random(77)
    sets = [W.make_patterns(3000, 0xAC5000), W.make_patterns(50, 0xAC0050),
            [b"a", b"ab", b"abc", b"b", b"bca", b"a"], [b"Sam", b"Samwise", b"sam", b"wise"]]
    for _ in range(40):
        n = rng.randint(1, 40)
        sets.append([bytes(rng.choice(b"abAB") for _ in range(rng.randint(1, 6))) for _ in range(n)])
    for pats in sets:
        for kind in (0, 1, 2):
            for ci in (False, True):
                built = (ab.AhoCorasick.builder().match_kind(kind).ascii_case_insensitive(ci)
                         .kind(ab.AhoCorasickKind.DFA).host_only(True).build(pats))
                t = built.tables()
                t["start_kind"] = 0
                adopted = _adopt(t)
                pb, pa = plan_of(built), plan_of(adopted)
                assert pb.n_rows == pa.n_rows
                db = np.ctypeslib.as_array(pb.depth16, shape=(pb.n_rows,))
                da = np.ctypeslib.as_array(pa.depth16, shape=(pa.n_rows,))
                assert np.array_equal(db, da), (pats[:5], kind, ci)
