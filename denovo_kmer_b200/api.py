"""Host-side mirror of the hot path's operator surface, over the C ABI only.

Names follow the reference's domain (north_star: src/kmer.rs, src/counter.rs — not in
the mount, DESIGN.md §2 is the spec): k-mers, spanning k-mer entries, read streams,
per-sample counts, de novo calls.  Everything that computes goes through libdkb.so;
there is no NumPy/PyTorch compute path here.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import Stats, Thresholds, Tuning, check, u8p, u16p, u32p, u64p

CHILD, MOTHER, FATHER = 0, 1, 2
REF, ALT = 0, 1
CALL_DENOVO, CALL_CHILD_LOW, CALL_MOTHER_ALT, CALL_FATHER_ALT, CALL_PARENT_UNCOVERED, CALL_NO_COPY = (
    0x01, 0x02, 0x04, 0x08, 0x10, 0x20)
# locus class of a variant (set_locus_classes) and sex of a child (set_child_sexes)
LOCUS_AUTOSOMAL, LOCUS_X, LOCUS_Y, LOCUS_MATERNAL = 0, 1, 2, 3
SEX_UNKNOWN, SEX_MALE, SEX_FEMALE = 0, 1, 2
DEFAULT_THRESHOLDS = (3, 2, 0, 1)
DEFAULT_MIN_BASEQ = 20
MAX_CHILDREN = _lib.MAX_CHILDREN


def _p(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def comm_unique_id() -> bytes:
    """Rank 0: the 128-byte NCCL id every rank passes to KmerCounter.comm_init."""
    buf = C.create_string_buffer(_lib.COMM_ID_BYTES)
    check(_lib.lib().dkb_comm_unique_id(buf))
    return buf.raw


# ---- kmer.rs primitives -----------------------------------------------------------
def kmer_encode(seq: str, k: int = None) -> int:
    k = len(seq) if k is None else k
    out = C.c_uint64(0)
    check(_lib.lib().dkb_kmer_encode(seq.encode(), k, C.byref(out)))
    return int(out.value)


def kmer_revcomp(fwd: int, k: int) -> int:
    return int(_lib.lib().dkb_kmer_revcomp(int(fwd), k))


def kmer_canonical(fwd: int, k: int) -> int:
    return int(_lib.lib().dkb_kmer_canonical(int(fwd), k))


# ---- packed read stream -------------------------------------------------------------
@dataclass
class ReadStream:
    """2-bit bases + 1-bit validity flags with one flag-0 separator after every read."""
    bases2: np.ndarray  # uint32
    mask1: np.ndarray   # uint32
    n_positions: int
    n_bases: int        # read bases only (the throughput unit), separators excluded


def stream_words(n_positions: int):
    L = _lib.lib()
    return int(L.dkb_stream_bases_words(n_positions)), int(L.dkb_stream_mask_words(n_positions))


def pack_reads(seq, qual, offsets, min_baseq: int = DEFAULT_MIN_BASEQ, pinned: bool = False,
               four_bit: bool = False):
    """seq/qual: uint8 arrays of concatenated reads (qual may be None);
    offsets: uint64[n_reads + 1] (in bases).  four_bit: seq holds BAM 4-bit codes, high nibble
    first, every read on a byte boundary (include/dkb.h, dkb_pack_reads_fmt) instead of ASCII.
    Returns a ReadStream in host memory."""
    L = _lib.lib()
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    qual = None if qual is None else np.ascontiguousarray(qual, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n_reads = len(offsets) - 1
    n_pos = int(L.dkb_stream_positions(_p(offsets, u64p), n_reads))
    bw, mw = stream_words(n_pos)
    if pinned:
        import torch
        tb = torch.empty(max(bw, 1), dtype=torch.int32).pin_memory()
        tm = torch.empty(max(mw, 1), dtype=torch.int32).pin_memory()
        bases2 = tb.numpy().view(np.uint32)
        mask1 = tm.numpy().view(np.uint32)
    else:
        bases2 = np.empty(max(bw, 1), dtype=np.uint32)
        mask1 = np.empty(max(mw, 1), dtype=np.uint32)
    out = C.c_uint64(0)
    check(L.dkb_pack_reads_fmt(_p(seq, u8p), int(four_bit), _p(qual, u8p), _p(offsets, u64p), n_reads,
                               min_baseq, _p(bases2, u32p), _p(mask1, u32p), C.byref(out)))
    n_bases = int(offsets[-1] - offsets[0]) if n_reads else 0
    return ReadStream(bases2, mask1, int(out.value), n_bases)


def mask_to_zero_list(mask1, n_positions: int):
    """Dense flags -> zero list (include/dkb.h): (zoff uint32[n_blocks + 1], zbytes uint8[used])."""
    L = _lib.lib()
    mask1 = np.ascontiguousarray(mask1).view(np.uint32)
    nb = int(L.dkb_zero_list_blocks(n_positions))
    zoff = np.zeros(nb + 1, dtype=np.uint32)
    used = C.c_size_t(0)
    # one call: a zero list is never longer than the dense flags (256 bytes per 2048-position block)
    zbytes = np.empty(max(nb * 256, 1), dtype=np.uint8)
    check(L.dkb_mask_to_zero_list(_p(mask1, u32p), n_positions, _p(zoff, u32p), _p(zbytes, u8p),
                                  len(zbytes), C.byref(used)))
    return zoff, zbytes[: int(used.value)]


# ---- spanning k-mer entries -----------------------------------------------------------
@dataclass
class KmerEntries:
    keys: np.ndarray       # uint64 canonical
    variant: np.ndarray    # uint32
    allele: np.ndarray     # uint8
    win_index: np.ndarray = None  # uint16 (bit 15: haplotype window is the key's rc)
    win_count: np.ndarray = None  # uint16
    n_variants: int = 0

    def __len__(self):
        return len(self.keys)


def variant_kmers(variants, k: int, drop_shared: bool = True) -> KmerEntries:
    """variants: sequence of (left_flank, ref, alt, right_flank) strings."""
    L = _lib.lib()
    n = len(variants)
    arrs = []
    for col in range(4):
        a = (C.c_char_p * max(n, 1))()
        for i, v in enumerate(variants):
            a[i] = v[col].encode()
        arrs.append(a)
    n_out = C.c_size_t(0)
    check(L.dkb_variant_kmers(*arrs, n, k, int(drop_shared), None, None, None, None, None,
                              C.byref(n_out)))
    m = int(n_out.value)
    keys = np.zeros(max(m, 1), dtype=np.uint64)
    var = np.zeros(max(m, 1), dtype=np.uint32)
    al = np.zeros(max(m, 1), dtype=np.uint8)
    wi = np.zeros(max(m, 1), dtype=np.uint16)
    wc = np.zeros(max(m, 1), dtype=np.uint16)
    check(L.dkb_variant_kmers(*arrs, n, k, int(drop_shared), _p(keys, u64p), _p(var, u32p),
                              _p(al, u8p), _p(wi, u16p), _p(wc, u16p), C.byref(n_out)))
    return KmerEntries(keys[:m], var[:m], al[:m], wi[:m], wc[:m], n)


# ---- region mode (include/dkb.h "region-scoped counting") ------------------------------------
@dataclass
class ReadLoci:
    """Where a batch's reads aligned: offsets as given to the packer (uint64[n_reads + 1]), and
    each read's half-open alignment interval [lo, hi) in the caller's linear coordinates
    (lo >= hi: unmapped, counts toward nothing)."""
    offsets: np.ndarray
    lo: np.ndarray
    hi: np.ndarray

    def __post_init__(self):
        self.offsets = np.ascontiguousarray(self.offsets, dtype=np.uint64)
        self.lo = np.ascontiguousarray(self.lo, dtype=np.uint64)
        self.hi = np.ascontiguousarray(self.hi, dtype=np.uint64)
        n = len(self.offsets) - 1
        if n < 0 or len(self.lo) != n or len(self.hi) != n:
            raise ValueError("ReadLoci: lo and hi need one entry per read (len(offsets) - 1)")


# ---- the counter -----------------------------------------------------------------------
def child_sample(c: int) -> int:
    """Sample index of child c of a family (DKB_CHILD_SAMPLE): 0 for c == 0, else 2 + c; the
    mother stays 1 and the father 2."""
    return 0 if c == 0 else c + 2


class KmerCounter:
    """One GPU context: build the spanning-k-mer table, stream read batches per
    sample, fetch per-entry / per-variant counts and de novo calls.

    n_children > 1 makes a family context: the mother (sample 1), the father (sample 2) and
    n_children children (sample child_sample(c)) counted against one table, n_samples =
    2 + n_children, and the de novo rule applied once per child."""

    def __init__(self, k: int, device: int = 0, tuning=None, n_children: int = 1):
        self._L = _lib.lib()
        self._h = C.c_void_p()
        self.k = k
        self.device = device
        self.n_children = int(n_children)
        self.n_samples = 2 + self.n_children
        check(self._L.dkb_ctx_create_family(device, k, self.n_children, C.byref(self._h)))
        if tuning is not None:
            self.set_tuning(*tuning)
        self.n_entries = 0
        self.n_variants = 0
        self._keep = []  # host buffers of in-flight submits
        self._pinned = []  # dkb_host_alloc blocks

    child_sample = staticmethod(child_sample)

    def close(self):
        if getattr(self, "_h", None):
            self._L.dkb_sync(self._h)
            for p in self._pinned:
                self._L.dkb_host_free(self._h, p)
            self._pinned = []
            self._L.dkb_ctx_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, code):
        check(code, self._h)

    def set_tuning(self, seed_len=0, stride=0, bloom_hashes=0, filter_mode=0):
        """0 = auto for every field; filter_mode 1 = shared memory, 2 = L2 (with or without the
        shared-memory pre-filter: the library's choice)."""
        t = Tuning(seed_len, stride, bloom_hashes, filter_mode)
        self._ck(self._L.dkb_ctx_set_tuning(self._h, C.byref(t)))

    def tuning(self):
        t = Tuning()
        self._ck(self._L.dkb_ctx_get_tuning(self._h, C.byref(t)))
        return t.seed_len, t.stride, t.bloom_hashes, t.filter_mode

    def build_table(self, entries: KmerEntries, use_window_hints: bool = True):
        keys = np.ascontiguousarray(entries.keys, dtype=np.uint64)
        var = np.ascontiguousarray(entries.variant, dtype=np.uint32)
        al = np.ascontiguousarray(entries.allele, dtype=np.uint8)
        wi = wc = None
        if use_window_hints and entries.win_index is not None and entries.win_count is not None:
            wi = np.ascontiguousarray(entries.win_index, dtype=np.uint16)
            wc = np.ascontiguousarray(entries.win_count, dtype=np.uint16)
        self._ck(self._L.dkb_table_build(self._h, _p(keys, u64p), _p(var, u32p), _p(al, u8p),
                                         _p(wi, u16p), _p(wc, u16p), len(keys),
                                         int(entries.n_variants)))
        self.n_entries = len(keys)
        self.n_variants = int(entries.n_variants)

    def set_regions(self, lo, hi):
        """Region mode: from now on a read's k-mers count toward variant v only if the read's
        alignment interval overlaps [lo[v], hi[v]) (one entry per variant of the table; lo >= hi:
        nothing counts toward v).  Every submit then needs loci=ReadLoci(...)."""
        lo = np.ascontiguousarray(lo, dtype=np.uint64)
        hi = np.ascontiguousarray(hi, dtype=np.uint64)
        if len(lo) != len(hi):
            raise ValueError("set_regions: lo and hi differ in length")
        self._ck(self._L.dkb_table_set_regions(self._h, _p(lo, u64p), _p(hi, u64p), len(lo)))

    def clear_regions(self):
        """Back to whole-stream counting."""
        self._ck(self._L.dkb_table_set_regions(self._h, None, None, 0))

    def set_locus_classes(self, cls):
        """Locus class of every variant of the table (LOCUS_AUTOSOMAL - PARs included -,
        LOCUS_X, LOCUS_Y outside the PARs, LOCUS_MATERNAL for MT): from now on a call applies
        only the clauses of the parents who can transmit the variant's locus to the child
        (include/dkb.h "inheritance").  A new table returns to all autosomal."""
        cls = np.ascontiguousarray(cls, dtype=np.uint8)
        self._ck(self._L.dkb_table_set_locus_classes(self._h, _p(cls, u8p), len(cls)))

    def clear_locus_classes(self):
        """Back to every variant autosomal."""
        self._ck(self._L.dkb_table_set_locus_classes(self._h, None, 0))

    def set_child_sexes(self, sexes):
        """Sex of every child (SEX_UNKNOWN, SEX_MALE, SEX_FEMALE; one per child); None returns
        every child to unknown.  Kept across table builds."""
        if sexes is None:
            self._ck(self._L.dkb_ctx_set_child_sexes(self._h, None, 0))
            return
        sx = np.ascontiguousarray(sexes, dtype=np.uint8)
        self._ck(self._L.dkb_ctx_set_child_sexes(self._h, _p(sx, u8p), len(sx)))

    def _set_loci(self, loci):
        if loci is None:
            return
        self._keep.append(loci)
        self._ck(self._L.dkb_batch_set_loci(self._h, _p(loci.offsets, u64p), _p(loci.lo, u64p),
                                            _p(loci.hi, u64p), len(loci.offsets) - 1))

    def submit(self, stream: ReadStream, sample: int, loci: ReadLoci = None):
        """Host buffers: async H2D copy + scan; buffers are kept alive until sync().
        loci: the batch's read loci (region mode)."""
        self._set_loci(loci)
        self._keep.append(stream)
        self._ck(self._L.dkb_batch_submit(self._h, stream.bases2.ctypes.data,
                                          stream.mask1.ctypes.data, stream.n_positions, sample))

    def submit_sparse(self, bases2, zoff, zbytes, n_positions: int, sample: int, loci: ReadLoci = None):
        """Host buffers with the flags as a zero list (mask_to_zero_list): less PCIe traffic."""
        self._set_loci(loci)
        self._keep.append((bases2, zoff, zbytes))
        self._ck(self._L.dkb_batch_submit_sparse(self._h, bases2.ctypes.data, zoff.ctypes.data,
                                                 zbytes.ctypes.data, len(zbytes), n_positions, sample))

    def submit_reads(self, seq, qual, offsets, sample: int, min_baseq: int = DEFAULT_MIN_BASEQ,
                     four_bit: bool = False, loci: ReadLoci = None):
        """Decoded reads (ASCII, or BAM 4-bit codes when four_bit) packed on the GPU."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        qual = None if qual is None else np.ascontiguousarray(qual, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self._set_loci(loci)
        self._keep.append((seq, qual, offsets))
        self._ck(self._L.dkb_batch_submit_reads(
            self._h, seq.ctypes.data, int(four_bit), None if qual is None else qual.ctypes.data,
            offsets.ctypes.data, len(offsets) - 1, min_baseq, sample))

    def submit_device(self, d_bases2: int, d_mask1: int, n_positions: int, sample: int,
                      loci: ReadLoci = None):
        """Device pointers (ints) of a resident stream.  loci stay referenced until sync()."""
        self._set_loci(loci)
        self._ck(self._L.dkb_batch_submit_device(self._h, d_bases2, d_mask1, n_positions, sample))

    def _set_loci_multi(self, loci, n):
        if loci is None:
            return
        if len(loci) != n:
            raise ValueError("loci: one ReadLoci per batch")
        self._keep.append(loci)
        arr = lambda f: (u64p * n)(*[_p(getattr(x, f), u64p) for x in loci])  # noqa: E731
        nr = (C.c_size_t * n)(*[len(x.offsets) - 1 for x in loci])
        self._ck(self._L.dkb_batch_set_loci_multi(self._h, n, arr("offsets"), arr("lo"), arr("hi"), nr))

    def submit_multi(self, streams, samples, loci=None):
        """Up to 4 host streams (ReadStream) scanned in ONE kernel launch, streams[i] into the
        counters of samples[i] (e.g. the three samples of a trio step).  loci: region mode, one
        ReadLoci per stream.  Buffers are kept alive until sync()."""
        n = len(streams)
        if len(samples) != n:
            raise ValueError("submit_multi: one sample per stream")
        self._set_loci_multi(loci, n)
        self._keep.append(streams)
        b = (C.c_void_p * n)(*[s.bases2.ctypes.data for s in streams])
        m = (C.c_void_p * n)(*[s.mask1.ctypes.data for s in streams])
        npos = (C.c_uint64 * n)(*[int(s.n_positions) for s in streams])
        smp = (C.c_int * n)(*[int(x) for x in samples])
        self._ck(self._L.dkb_batch_submit_multi(self._h, n, b, m, npos, smp))

    def submit_sparse_multi(self, batches, samples, loci=None):
        """Up to 4 host batches with their flags as zero lists (mask_to_zero_list), expanded by
        one launch and scanned by one: batches[i] = (bases2, zoff, zbytes, n_positions) goes into
        the counters of samples[i].  loci: region mode, one ReadLoci per batch.  Buffers are kept
        alive until sync()."""
        n = len(batches)
        if len(samples) != n:
            raise ValueError("submit_sparse_multi: one sample per batch")
        batches = [(np.ascontiguousarray(b, dtype=np.uint32), np.ascontiguousarray(z, dtype=np.uint32),
                    np.ascontiguousarray(zb, dtype=np.uint8), int(npos)) for b, z, zb, npos in batches]
        self._set_loci_multi(loci, n)
        self._keep.append(batches)
        ptrs = lambda j: (C.c_void_p * n)(*[x[j].ctypes.data for x in batches])  # noqa: E731
        used = (C.c_size_t * n)(*[len(x[2]) for x in batches])
        npos = (C.c_uint64 * n)(*[x[3] for x in batches])
        smp = (C.c_int * n)(*[int(x) for x in samples])
        self._ck(self._L.dkb_batch_submit_sparse_multi(self._h, n, ptrs(0), ptrs(1), ptrs(2), used, npos, smp))

    def submit_reads_multi(self, reads, samples, min_baseq: int = DEFAULT_MIN_BASEQ, four_bit: bool = False,
                           loci=None):
        """Up to 4 batches of decoded reads (ASCII, or BAM 4-bit codes when four_bit) packed by
        one launch and scanned by one: reads[i] = (seq, qual, offsets), qual may be None, goes
        into the counters of samples[i].  loci: region mode, one ReadLoci per batch.  Buffers
        are kept alive until sync()."""
        n = len(reads)
        if len(samples) != n:
            raise ValueError("submit_reads_multi: one sample per batch")
        reads = [(np.ascontiguousarray(s, dtype=np.uint8), None if q is None else np.ascontiguousarray(q, dtype=np.uint8),
                  np.ascontiguousarray(o, dtype=np.uint64)) for s, q, o in reads]
        self._set_loci_multi(loci, n)
        self._keep.append(reads)
        seq = (C.c_void_p * n)(*[x[0].ctypes.data for x in reads])
        qual = (C.c_void_p * n)(*[None if x[1] is None else x[1].ctypes.data for x in reads])
        offs = (C.c_void_p * n)(*[x[2].ctypes.data for x in reads])
        nr = (C.c_size_t * n)(*[len(x[2]) - 1 for x in reads])
        smp = (C.c_int * n)(*[int(x) for x in samples])
        self._ck(self._L.dkb_batch_submit_reads_multi(self._h, n, seq, int(four_bit), qual, offs, nr, min_baseq,
                                                      smp))

    def submit_device_multi(self, batches, loci=None):
        """batches: up to 4 tuples (d_bases2, d_mask1, n_positions, sample) of resident
        streams, scanned in ONE kernel launch (e.g. the three samples of a trio, or the four of
        a quad).  loci: region mode, one ReadLoci per batch, referenced until sync()."""
        n = len(batches)
        self._set_loci_multi(loci, n)
        b = (C.c_void_p * n)(*[int(x[0]) for x in batches])
        m = (C.c_void_p * n)(*[int(x[1]) for x in batches])
        npos = (C.c_uint64 * n)(*[int(x[2]) for x in batches])
        smp = (C.c_int * n)(*[int(x[3]) for x in batches])
        self._ck(self._L.dkb_batch_submit_device_multi(self._h, n, b, m, npos, smp))

    def sync(self):
        self._ck(self._L.dkb_sync(self._h))
        self._keep.clear()

    def reset_counts(self):
        self._ck(self._L.dkb_counts_reset(self._h))

    def entry_counts(self) -> np.ndarray:
        """[n_samples, n_entries] per-entry counters."""
        out = np.zeros((self.n_samples, max(self.n_entries, 1)), dtype=np.uint32)
        self._ck(self._L.dkb_entry_counts_fetch(self._h, _p(out, u32p)))
        self._keep.clear()
        return out[:, : self.n_entries]

    def entry_counts_device(self):
        """(device pointer, number of uint32) of the [n_samples][n_entries] counters."""
        p = C.c_void_p()
        n = C.c_size_t(0)
        self._ck(self._L.dkb_entry_counts_device(self._h, C.byref(p), C.byref(n)))
        return int(p.value or 0), int(n.value)

    def finalise_launch(self, thresholds=DEFAULT_THRESHOLDS, counts_ptr=None):
        """Queue kernel 3 on the scan stream without waiting for it.  counts_ptr: device
        pointer of a caller-owned copy of the [n_samples][n_entries] counters (dkb_finalise_from)."""
        t = Thresholds(*[int(x) for x in thresholds])
        if counts_ptr is None:
            self._ck(self._L.dkb_finalise(self._h, C.byref(t)))
        else:
            self._ck(self._L.dkb_finalise_from(self._h, C.byref(t), C.c_void_p(int(counts_ptr))))

    def finalise(self, thresholds=DEFAULT_THRESHOLDS):
        """Kernel 3 + fetch: (hits[nv,2,n_samples], distinct[nv,2,n_samples], n_kmers[nv,2],
        calls[nv] for a trio or calls[nv,n_children] for a family)."""
        self.finalise_launch(thresholds)
        return self.results()

    def results(self):
        """(hits, distinct, n_kmers, calls) of the last finalise; shapes as in finalise()."""
        nv = max(self.n_variants, 1)
        hits = np.zeros((nv, 2, self.n_samples), dtype=np.uint32)
        dist = np.zeros((nv, 2, self.n_samples), dtype=np.uint32)
        nk = np.zeros((nv, 2), dtype=np.uint32)
        calls = np.zeros((nv, self.n_children) if self.n_children > 1 else nv, dtype=np.uint8)
        self._ck(self._L.dkb_results_fetch(self._h, _p(hits, u32p), _p(dist, u32p), _p(nk, u32p),
                                           _p(calls, u8p)))
        self._keep.clear()  # the fetch waited for the scan stream: every submit has been consumed
        n = self.n_variants
        return hits[:n], dist[:n], nk[:n], calls[:n]

    # ---- pinned staging next to the GPU -----------------------------------------------------
    def host_alloc(self, n_words: int) -> np.ndarray:
        """uint32[n_words] in page-locked memory on the GPU's NUMA node (dkb_host_alloc); freed
        when the counter is closed."""
        p = C.c_void_p()
        self._ck(self._L.dkb_host_alloc(self._h, max(n_words, 1) * 4, C.byref(p)))
        self._pinned.append(p)
        return np.ctypeslib.as_array(C.cast(p, u32p), shape=(max(n_words, 1),))[:n_words]

    def bind_thread_near_gpu(self) -> int:
        """Pin the calling thread to the CPUs of the GPU's NUMA node; returns the node (-1 unknown)."""
        node = C.c_int(-1)
        self._ck(self._L.dkb_thread_bind_near_gpu(self._h, C.byref(node)))
        return node.value

    # ---- multi-GPU (include/dkb.h "multi-GPU"): NCCL inside the library ------------------
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        assert len(unique_id) == _lib.COMM_ID_BYTES
        buf = C.create_string_buffer(bytes(unique_id), _lib.COMM_ID_BYTES)
        self._ck(self._L.dkb_comm_init(self._h, buf, rank, world))

    def comm_destroy(self):
        self._ck(self._L.dkb_comm_destroy(self._h))

    def comm_info(self):
        """(rank, communicator size as NCCL reports it, NCCL version code)"""
        r, w, v = C.c_int(0), C.c_int(0), C.c_int(0)
        self._ck(self._L.dkb_comm_info(self._h, C.byref(r), C.byref(w), C.byref(v)))
        return r.value, w.value, v.value

    def counts_allreduce(self):
        """In-place sum over ranks of the counters, on the scan stream."""
        self._ck(self._L.dkb_counts_allreduce(self._h))

    def reduce_push(self, thresholds=DEFAULT_THRESHOLDS):
        """Snapshot the counters and start their sum over ranks on a side stream; queues
        kernel 3 for the PREVIOUS snapshot behind the scans submitted since.  The snapshot keeps
        the locus classes and child sexes in force now; its kernel 3 uses those."""
        t = Thresholds(*[int(x) for x in thresholds])
        self._ck(self._L.dkb_reduce_push(self._h, C.byref(t)))

    def reduce_flush(self, thresholds=DEFAULT_THRESHOLDS):
        t = Thresholds(*[int(x) for x in thresholds])
        self._ck(self._L.dkb_reduce_flush(self._h, C.byref(t)))

    def reduced_counts(self) -> np.ndarray:
        """Summed counters of the most recently finalised snapshot, [n_samples, n_entries]."""
        out = np.zeros((self.n_samples, max(self.n_entries, 1)), dtype=np.uint32)
        self._ck(self._L.dkb_reduced_counts_fetch(self._h, _p(out, u32p)))
        return out[:, : self.n_entries]

    def stats(self) -> dict:
        s = Stats()
        self._ck(self._L.dkb_stats_get(self._h, C.byref(s)))
        return {f: getattr(s, f) for f, _ in Stats._fields_}

    def profile_counters(self, enable: bool):
        self._ck(self._L.dkb_profile_counters(self._h, int(enable)))

    def scan_stream(self) -> int:
        p = C.c_void_p()
        self._ck(self._L.dkb_scan_stream(self._h, C.byref(p)))
        return int(p.value or 0)
