"""Test infrastructure for region-scoped counting (DESIGN.md §2): the C stream walk with read
loci (region_oracle.c, built on first use into a temporary directory) and a pure-Python
per-variant fetch - for every variant, take the reads whose alignment overlaps its window and
count that variant's live entries in those reads only, the way a tool that fetches reads per
candidate region counts.  The two share no logic; the tests pin one against the other, and
the GPU against the C walk."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "region_oracle.c")
_lib = None

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        so = os.path.join(tempfile.gettempdir(), f"dkb_region_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O3", "-fopenmp", "-fPIC", "-shared", "-Wall", "-std=c11", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_count_stream_loci.restype = C.c_int
        L.orc_count_stream_loci.argtypes = [u64p, u32p, u8p, C.c_size_t, u64p, u64p, u32p, u32p, C.c_uint64,
                                            u64p, u64p, u64p, C.c_size_t, C.c_int, u64p, C.c_int]
        _lib = L
    return _lib


def _a(x, t):
    return np.ascontiguousarray(x, dtype=t)


def count_stream_loci(keys, variant, allele, vlo, vhi, bases2, mask1, n_positions, offsets, rlo, rhi, k,
                      counts=None, threads=0):
    """Per-entry counts (uint64, added to `counts`) of one packed stream in region mode."""
    keys, variant, allele = _a(keys, np.uint64), _a(variant, np.uint32), _a(allele, np.uint8)
    vlo, vhi = _a(vlo, np.uint64), _a(vhi, np.uint64)
    offsets, rlo, rhi = _a(offsets, np.uint64), _a(rlo, np.uint64), _a(rhi, np.uint64)
    bases2 = np.ascontiguousarray(bases2).view(np.uint32)
    mask1 = np.ascontiguousarray(mask1).view(np.uint32)
    n_reads = len(offsets) - 1
    assert len(rlo) == n_reads and len(rhi) == n_reads
    assert int(offsets[-1] - offsets[0]) + n_reads == n_positions
    if counts is None:
        counts = np.zeros(len(keys), dtype=np.uint64)
    P = lambda a, t: a.ctypes.data_as(t)  # noqa: E731
    rc = lib().orc_count_stream_loci(P(keys, u64p), P(variant, u32p), P(allele, u8p), len(keys), P(vlo, u64p),
                                     P(vhi, u64p), P(bases2, u32p), P(mask1, u32p), int(n_positions),
                                     P(offsets, u64p), P(rlo, u64p), P(rhi, u64p), n_reads, k,
                                     P(counts, u64p), threads)
    assert rc == 0
    return counts


def windows(variants, pad, n_extra=0):
    """[pos - pad, pos + len(ref) + pad) per variant (clamped at 0), plus n_extra empty ones."""
    lo = np.array([max(0, v.pos - pad) for v in variants] + [0] * n_extra, dtype=np.uint64)
    hi = np.array([v.pos + len(v.ref) + pad for v in variants] + [0] * n_extra, dtype=np.uint64)
    return lo, hi


def py_fetch_counts(keys, variant, allele, n_variants, vlo, vhi, reads, k, min_bq=0):
    """Per-variant fetch in plain Python.  reads: per sample a list of (seq str, qual|None, lo,
    hi).  Returns uint64 [3, n_entries]."""
    import oracle
    n = len(keys)
    first, live = set(), np.zeros(n, dtype=bool)
    for i in range(n):
        t = (int(keys[i]), int(variant[i]), int(allele[i]))
        if t not in first:
            first.add(t)
            live[i] = True
    by_var = [dict() for _ in range(n_variants)]  # variant -> key -> live entries
    for i in np.nonzero(live)[0]:
        by_var[int(variant[i])].setdefault(int(keys[i]), []).append(int(i))
    out = np.zeros((3, n), dtype=np.uint64)
    for smp in range(3):
        kmers = [[key for _, key in oracle.py_read_kmers(seq, qual, k, min_bq)] for seq, qual, _, _ in reads[smp]]
        span = np.array([(lo, hi) for _, _, lo, hi in reads[smp]], dtype=np.uint64).reshape(-1, 2)
        for v in range(n_variants):
            a, b = int(vlo[v]), int(vhi[v])
            if a >= b or not by_var[v]:
                continue
            fetched = np.nonzero((span[:, 0] < span[:, 1]) & (span[:, 0] < b) & (span[:, 1] > a))[0]
            for r in fetched:
                for key in kmers[r]:
                    for e in by_var[v].get(key, ()):
                        out[smp, e] += 1
    return out


def trio_reads(trio, smp):
    """(seq str, qual, lo, hi) per read of one sample of a synth trio."""
    seq, qual, off = trio.reads[smp]
    lo, hi = trio.loci[smp]
    return [(seq[int(off[r]):int(off[r + 1])].tobytes().decode(), qual[int(off[r]):int(off[r + 1])],
             int(lo[r]), int(hi[r])) for r in range(len(off) - 1)]
