"""CPU: the de novo rule with inheritance (DESIGN.md §2 "Inheritance") - hand-derived bytes for
every (locus class, child sex) cell and clause, the C restatement against its pure-Python twin,
today's rule when everything is autosomal, the planted scenarios of make_sexed_family_host in
the oracle, and the new calls in every binding."""
import inspect
import os
import re

import numpy as np
import pytest

import inherit_oracle as io
from denovo_kmer_b200 import synth
from family_oracle import family_counts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K, THR, MIN_BQ = 31, (3, 2, 0, 1), 20
A, X, Y, MT = io.AUTOSOMAL, io.X, io.Y, io.MATERNAL
U, M, F = io.UNKNOWN, io.MALE, io.FEMALE

# Which parents' clauses apply, copied from the table of DESIGN.md §2 ("-": neither, no copy)
TABLE = {
    (A, U): "MF", (A, M): "MF", (A, F): "MF",
    (X, U): "MF", (X, M): "M", (X, F): "MF",
    (Y, U): "MF", (Y, M): "F", (Y, F): "-",
    (MT, U): "M", (MT, M): "M", (MT, F): "M",
}

# One candidate per failing clause: hits / distinct [2 alleles][child, mother, father] that pass
# every clause but the named one.  name -> (hits edit, distinct edit, bit, parent it belongs to);
# an edit is ((allele, sample), value).
GOOD_H, GOOD_D = [[0, 5, 5], [6, 0, 0]], [[0, 2, 2], [3, 0, 0]]
CLAUSES = {
    "none": (None, None, 0x00, None),
    "child_hits": (((1, 0), 2), None, 0x02, None),
    "child_distinct": (None, ((1, 0), 1), 0x02, None),
    "mother_alt": (((1, 1), 1), None, 0x04, "M"),
    "father_alt": (((1, 2), 1), None, 0x08, "F"),
    "mother_ref": (((0, 1), 0), None, 0x10, "M"),
    "father_ref": (((0, 2), 0), None, 0x10, "F"),
}


def _case(clause):
    h, d = np.array(GOOD_H, dtype=np.uint64), np.array(GOOD_D, dtype=np.uint64)
    for arr, edit in ((h, CLAUSES[clause][0]), (d, CLAUSES[clause][1])):
        if edit:
            arr[edit[0]] = edit[1]
    return h, d


def _hand_byte(cls, sex, clause):
    who = TABLE[(cls, sex)]
    _, _, bit, parent = CLAUSES[clause]
    applies = parent is None or parent in who
    c = (bit if applies else 0) | (0x20 if who == "-" else 0)
    return c or 0x01


CELLS = sorted(TABLE)


def test_hand_derived_bytes_trio():
    """Every cell times every clause: the C oracle and the Python twin give the hand-derived byte."""
    n = 0
    for cls, sex in CELLS:
        for clause in CLAUSES:
            h, d = _case(clause)
            want = _hand_byte(cls, sex, clause)
            got = io.calls(h[None], d[None], THR, np.array([cls], np.uint8), sex)
            assert got[0] == want, (cls, sex, clause, hex(got[0]), hex(want))
            assert io.py_calls(h[None], d[None], THR, [cls], sex)[0] == want
            n += 1
    assert n == 12 * len(CLAUSES)
    # a daughter at Y is never a call, whatever the counts
    assert _hand_byte(Y, F, "none") == 0x20


def test_hand_derived_bytes_family_layout():
    """The same cases laid out as a six-child family: child c's calls come from the rows
    [child_sample(c), 1, 2]; each child has its own sex, every variant its own class."""
    sexes = [U, M, F, M, F, U]
    cases = [(cls, clause) for cls in (A, X, Y, MT) for clause in CLAUSES]
    ns = 2 + len(sexes)
    hits = np.zeros((len(cases), 2, ns), np.uint64)
    dist = np.zeros((len(cases), 2, ns), np.uint64)
    for v, (cls, clause) in enumerate(cases):
        h, d = _case(clause)
        for c in range(len(sexes)):
            rows = [synth.child_sample(c), 1, 2]
            hits[v][:, rows], dist[v][:, rows] = h, d
    classes = np.array([cls for cls, _ in cases], np.uint8)
    for c, sex in enumerate(sexes):
        rows = [synth.child_sample(c), 1, 2]
        got = io.calls(hits[:, :, rows], dist[:, :, rows], THR, classes, sex)
        want = [_hand_byte(cls, sex, clause) for cls, clause in cases]
        assert got.tolist() == want, c


@pytest.mark.parametrize("seed", range(4))
def test_c_oracle_equals_python_twin(seed):
    rng = np.random.default_rng(seed)
    nv = 3000
    hits = rng.integers(0, 5, size=(nv, 2, 3)).astype(np.uint64)
    dist = np.minimum(hits, rng.integers(0, 4, size=(nv, 2, 3))).astype(np.uint64)
    classes = rng.integers(0, 4, size=nv).astype(np.uint8)
    thr = tuple(int(t) for t in rng.integers(0, 4, size=4))
    seen = set()
    for sex in (U, M, F):
        got = io.calls(hits, dist, thr, classes, sex)
        assert np.array_equal(got, io.py_calls(hits, dist, thr, classes, sex))
        seen |= {(int(c), sex, int(b)) for c, b in zip(classes, got)}
        assert np.array_equal(io.calls(hits, dist, thr, None, sex), io.py_calls(hits, dist, thr, None, sex))
    assert {(c, sx) for c, sx, _ in seen} == set(TABLE)


def test_all_autosomal_is_todays_rule(orc):
    rng = np.random.default_rng(9)
    nv = 2000
    hits = rng.integers(0, 5, size=(nv, 2, 3)).astype(np.uint64)
    dist = np.minimum(hits, rng.integers(0, 4, size=(nv, 2, 3))).astype(np.uint64)
    today = orc.calls(hits, dist, THR)
    for sex in (U, M, F):
        assert np.array_equal(io.calls(hits, dist, THR, np.zeros(nv, np.uint8), sex), today)
        assert np.array_equal(io.calls(hits, dist, THR, None, sex), today)
    # unknown sex keeps today's rule on X and Y
    xy = rng.integers(1, 3, size=nv).astype(np.uint8)
    assert np.array_equal(io.calls(hits, dist, THR, xy, U), today)


def test_sexed_generator_is_seeded_and_sexed():
    a = synth.make_sexed_family_host([M, F], K, seed=4)
    b = synth.make_sexed_family_host([M, F], K, seed=4)
    for smp in a.reads:
        assert all(np.array_equal(x, y) for x, y in zip(a.reads[smp], b.reads[smp]))
    # reads per segment follow the copy numbers: a son has no second X, a daughter no Y
    def per_segment(smp):
        lo = a.loci[smp][0].astype(np.int64)
        return {cls: int(((lo >= s0) & (lo < s1)).sum()) for cls, (s0, s1) in a.segments.items()}
    mother, father, son, daughter = (per_segment(s) for s in (1, 2, 0, 3))
    assert mother[Y] == 0 and daughter[Y] == 0 and son[Y] > 0 and father[Y] > 0
    assert abs(son[X] * 2 - mother[X]) <= 2 and abs(daughter[X] - mother[X]) <= 2
    assert abs(father[X] - son[X]) <= 1 and abs(son[A] - mother[A]) <= 1
    assert len(a.scenarios) == len(a.variants) == len(a.classes)
    assert set(a.scenarios) == set(synth.SEXED_SCENARIOS)


@pytest.mark.parametrize("sexes", [[M], [F], [M, F]])
def test_planted_scenarios_in_the_oracle(dkb, orc, sexes):
    """Every scenario gives its designed byte with classes and sexes set; each one outside the
    autosomes gives some child a different byte without them (on X, a son), and the autosomal
    controls do not."""
    fam = synth.make_sexed_family_host(sexes, K, seed=11, err_rate=0.0)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    nc = len(sexes)
    ks, counts = family_counts(orc, entries, fam, K, MIN_BQ, 2 + nc)
    nv = len(fam.variants)
    calls = io.family_results(orc, ks, counts, nv, nc, THR, fam.classes, fam.sexes)[3]
    plain = io.family_results(orc, ks, counts, nv, nc, THR)[3]
    for v, name in enumerate(fam.scenarios):
        cls, son, daughter = synth.SEXED_SCENARIOS[name]
        want = [son if s == M else daughter for s in sexes]
        assert calls[v].tolist() == want, (name, calls[v], want)
        if cls == A:
            assert np.array_equal(plain[v], calls[v]), name
        elif cls != X or M in sexes:  # a daughter's X keeps both parents' clauses
            assert not np.array_equal(plain[v], calls[v]), name


def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def test_python_layer(dkb):
    for name in ("set_locus_classes", "clear_locus_classes", "set_child_sexes"):
        assert callable(getattr(dkb.KmerCounter, name)), name
    assert list(inspect.signature(dkb.KmerCounter.set_locus_classes).parameters) == ["self", "cls"]
    assert (dkb.LOCUS_AUTOSOMAL, dkb.LOCUS_X, dkb.LOCUS_Y, dkb.LOCUS_MATERNAL) == (0, 1, 2, 3)
    assert (dkb.SEX_UNKNOWN, dkb.SEX_MALE, dkb.SEX_FEMALE) == (0, 1, 2) and dkb.CALL_NO_COPY == 0x20
    from denovo_kmer_b200 import _lib
    for fn in ("dkb_table_set_locus_classes", "dkb_ctx_set_child_sexes"):
        assert fn in _lib.SYMBOLS


def test_header_constants():
    hdr = _read("include", "dkb.h")
    for name, val in (("DKB_CALL_NO_COPY", "0x20u"), ("DKB_LOCUS_AUTOSOMAL", "0"), ("DKB_LOCUS_X", "1"),
                      ("DKB_LOCUS_Y", "2"), ("DKB_LOCUS_MATERNAL", "3"), ("DKB_SEX_UNKNOWN", "0"),
                      ("DKB_SEX_MALE", "1"), ("DKB_SEX_FEMALE", "2")):
        assert re.search(rf"#define {name} {val}\b", hdr), name
    sysrs = _read("bindings", "rust", "denovo-kmer-gpu-sys", "src", "lib.rs")
    for name, val in (("DKB_CALL_NO_COPY", "0x20"), ("DKB_LOCUS_MATERNAL", "3"), ("DKB_SEX_FEMALE", "2")):
        assert f"pub const {name}: u8 = {val};" in sysrs, name


def test_cpp_layer_wraps_both_calls():
    hpp = _read("include", "dkb.hpp")
    for fn in ("dkb_table_set_locus_classes", "dkb_ctx_set_child_sexes"):
        assert re.search(r"check\(\s*" + fn + r"\(", hpp), fn
    for m in ("void set_locus_classes(", "void clear_locus_classes(", "void set_child_sexes("):
        assert m in hpp, m


def test_rust_safe_crate_calls_both():
    safe = _read("bindings", "rust", "denovo-kmer-gpu", "src", "lib.rs")
    assert re.search(r"pub fn set_locus_classes\(&mut self, cls: &\[LocusClass\]\)", safe)
    assert re.search(r"pub fn set_child_sexes\(&mut self, sexes: &\[Sex\]\)", safe)
    assert "sys::dkb_table_set_locus_classes(" in safe and "sys::dkb_ctx_set_child_sexes(" in safe
    assert re.search(r"pub enum LocusClass \{", safe) and re.search(r"pub enum Sex \{", safe)
