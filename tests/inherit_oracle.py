"""Test infrastructure for the de novo rule with inheritance (DESIGN.md §2 "Inheritance"): the C
restatement (inherit_oracle.c, built on first use into a temporary directory), a pure-Python
twin written from the transmission rules rather than the table, and the per-child family
results with locus classes and child sexes.  With no classes and unknown sexes, `calls` is the
trio oracle's `oracle.calls`."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from denovo_kmer_b200.synth import child_sample

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "inherit_oracle.c")
_lib = None

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)

AUTOSOMAL, X, Y, MATERNAL = 0, 1, 2, 3
UNKNOWN, MALE, FEMALE = 0, 1, 2
NO_COPY = 0x20


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        so = os.path.join(tempfile.gettempdir(), f"dkb_inherit_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-std=c11", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_calls_inherit.argtypes = [u64p, u64p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                        u8p, C.c_uint8, u8p]
        _lib = L
    return _lib


def calls(hits, distinct, thr, classes=None, sex=0):
    """Trio calls [nv] from hits / distinct [nv, 2, 3] (child, mother, father) under thresholds
    thr, for variants of locus classes `classes` (uint8 per variant; None = all autosomal) and a
    child of sex `sex`."""
    import oracle
    hits = np.ascontiguousarray(hits, dtype=np.uint64)
    distinct = np.ascontiguousarray(distinct, dtype=np.uint64)
    nv = hits.shape[0]
    if classes is None and sex == UNKNOWN:
        return oracle.calls(hits, distinct, thr)
    cls = None if classes is None else np.ascontiguousarray(classes, dtype=np.uint8)
    assert cls is None or len(cls) == nv
    out = np.zeros(max(nv, 1), dtype=np.uint8)
    P = lambda a, t: None if a is None else a.ctypes.data_as(t)  # noqa: E731
    lib().orc_calls_inherit(P(hits, u64p), P(distinct, u64p), nv, *[int(t) for t in thr], P(cls, u8p), int(sex),
                            P(out, u8p))
    return out[:nv]


def py_parents(cls, sex):
    """(mother's clauses apply, father's apply, the child has no copy) from who transmits what:
    the mother transmits an X to every child and the mitochondria to every child, the father
    an X to daughters only and a Y to sons only; an unknown sex keeps both parents on X and Y."""
    if cls == MATERNAL:
        return True, False, False
    if cls == X and sex == MALE:
        return True, False, False
    if cls == Y and sex == MALE:
        return False, True, False
    if cls == Y and sex == FEMALE:
        return False, False, True
    return True, True, False


def py_calls(hits, distinct, thr, classes=None, sex=0):
    """Pure-Python twin of `calls`."""
    min_alt, min_alt_d, max_parent_alt, min_parent_ref = (int(t) for t in thr)
    out = []
    for v in range(len(hits)):
        h, d = hits[v], distinct[v]
        mother, father, no_copy = py_parents(AUTOSOMAL if classes is None else int(classes[v]), sex)
        c = 0
        if h[1][0] < min_alt or d[1][0] < min_alt_d:
            c |= 0x02
        if mother and h[1][1] > max_parent_alt:
            c |= 0x04
        if father and h[1][2] > max_parent_alt:
            c |= 0x08
        if (mother and h[0][1] < min_parent_ref) or (father and h[0][2] < min_parent_ref):
            c |= 0x10
        if no_copy:
            c |= NO_COPY
        out.append(c or 0x01)
    return np.array(out, dtype=np.uint8)


def family_results(orc, ks, counts, n_variants, n_children, thr, classes=None, sexes=None):
    """tests/family_oracle.family_results with locus classes and each child's sex (sexes[c];
    None = all unknown): hits, distinct [nv, 2, NS], n_kmers [nv, 2], calls [nv, n_children]."""
    ns = 2 + n_children
    sexes = [UNKNOWN] * n_children if sexes is None else list(sexes)
    hits = np.zeros((n_variants, 2, ns), dtype=np.uint64)
    dist = np.zeros((n_variants, 2, ns), dtype=np.uint64)
    out = np.zeros((n_variants, n_children), dtype=np.uint8)
    nk = None
    for c in range(n_children):
        rows = [child_sample(c), 1, 2]
        h, d, nk = ks.variant_stats(counts[rows], n_variants)
        hits[:, :, rows] = h
        dist[:, :, rows] = d
        out[:, c] = calls(h, d, thr, classes, sexes[c])
    return hits, dist, nk, out
