"""-m gpu: the multi-batch forms of the zero-list and decoded-read transports -
dkb_batch_submit_sparse_multi and dkb_batch_submit_reads_multi (ASCII and BAM 4-bit) - expand or
pack up to four batches in one launch and scan them in one, and count exactly what the oracle
and one single-form submit per batch count: counters, positions scanned, hits / distinct /
calls, whole stream and region mode, over odd lengths, empty batches and reads, mask-word and
zero-list-block edges, plain-bits blocks, adversarial batch edges, pipelined submits that grow
the staging buffers, and every refusal."""
import ctypes as C

import numpy as np
import pytest

import adversarial as adv
import region_oracle as ro
from denovo_kmer_b200 import synth
from family_oracle import family_results
from test_gpu_multi_submit import THR, MIN_BQ, UNEVEN, _region_want, _split, _steps, _submit_step
from test_gpu_regions import TUNINGS, _four_bit, _trimmed

pytestmark = pytest.mark.gpu

FORMS = ("sparse", "reads", "reads4")


def _multi(dkb, kc, form, step, loci=None, min_bq=MIN_BQ):
    """One multi-batch submit of `step` ([(sample, stream, loci, seq, qual, off)]) in `form`."""
    samples = [b[0] for b in step]
    if form == "sparse":
        zl = [dkb.mask_to_zero_list(b[1].mask1, b[1].n_positions) for b in step]
        kc.submit_sparse_multi([(b[1].bases2, z[0], z[1], b[1].n_positions) for b, z in zip(step, zl)], samples,
                               loci=loci)
    elif form == "reads":
        kc.submit_reads_multi([(b[3], b[4], b[5]) for b in step], samples, min_bq, loci=loci)
    else:
        kc.submit_reads_multi([(_four_bit(b[3], b[5]), b[4], b[5]) for b in step], samples, min_bq, four_bit=True,
                              loci=loci)


def _single(dkb, kc, form, b, loci=None):
    """One single-form submit of batch b (its offsets start at 0)."""
    smp, st, _, seq, qual, off = b
    if form == "sparse":
        zoff, zbytes = dkb.mask_to_zero_list(st.mask1, st.n_positions)
        kc.submit_sparse(st.bases2, zoff, zbytes, st.n_positions, smp, loci=loci)
    elif form == "reads":
        kc.submit_reads(seq, qual, off, smp, MIN_BQ, loci=loci)
    else:
        kc.submit_reads(_four_bit(seq, off), qual, off, smp, MIN_BQ, four_bit=True, loci=loci)


def _counter_run(dkb, entries, k, submit_all, vlo=None, vhi=None, tuning=None, hints=True, n_children=1):
    with dkb.KmerCounter(k, tuning=tuning, n_children=n_children) as kc:
        kc.build_table(entries, use_window_hints=hints)
        if vlo is not None:
            kc.set_regions(vlo, vhi)
        s0 = kc.stats()
        submit_all(kc)
        kc.sync()
        st = kc.stats()
        got = kc.entry_counts().copy()
        res = kc.finalise(THR)
        tun = kc.tuning()
    return dict(counts=got, res=res, tuning=tun, launches=st["scan_launches"] - s0["scan_launches"],
                positions=st["positions_scanned"] - s0["positions_scanned"])


def _run_multi(dkb, entries, k, steps, form, regions=None, **kw):
    def go(kc):
        for step in steps:
            _multi(dkb, kc, form, step, [b[2] for b in step] if regions else None)
    return _counter_run(dkb, entries, k, go, *(regions or (None, None)), **kw)


def _run_single(dkb, entries, k, steps, form, regions=None, **kw):
    def go(kc):
        for step in steps:
            for b in step:
                _single(dkb, kc, form, b, b[2] if regions else None)
    return _counter_run(dkb, entries, k, go, *(regions or (None, None)), **kw)


def _check_forms(dkb, orc, entries, k, steps, ns, regions=None, forms=FORMS, **kw):
    """Every form's multi submits of `steps` equal the oracle and the same batches one single
    submit each; one scan launch per multi submit with positions."""
    batches = [b for step in steps for b in step]
    if regions:
        want = _region_want(orc, entries, batches, *regions, k, ns)
    else:
        ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
        want = np.zeros((ns, len(entries)), dtype=np.uint64)
        for smp, _, _, seq, qual, off in batches:
            if len(off) > 1:
                ks.count_reads(seq, qual, off, k, MIN_BQ, counts=want[smp])
    assert want.sum() > 0
    n_launch = sum(any(b[1].n_positions > 0 for b in step) for step in steps)
    n_pos = sum(int(b[1].n_positions) for b in batches)
    for form in forms:
        m = _run_multi(dkb, entries, k, steps, form, regions, **kw)
        bad = np.argwhere(m["counts"].astype(np.uint64) != want)
        assert len(bad) == 0, (form, m["tuning"], len(bad),
                               [(int(s), int(e), int(m["counts"][s, e]), int(want[s, e])) for s, e in bad[:5]])
        assert m["launches"] == n_launch, form
        assert m["positions"] == n_pos, form
        s = _run_single(dkb, entries, k, steps, form, regions, **kw)
        assert np.array_equal(s["counts"], m["counts"]) and s["positions"] == m["positions"], form
        for a, b in zip(s["res"], m["res"]):
            assert np.array_equal(a, b), form
    return want, m


def _noqual(dkb, b):
    """The batch without base qualities (qual NULL)."""
    smp, _, loci, seq, _, off = b
    return (smp, dkb.pack_reads(seq, None, off, MIN_BQ), loci, seq, None, off)


# ---- whole stream: a trio and a quad ------------------------------------------------------------
@pytest.mark.parametrize("n_children", [1, 2])
def test_trio_and_quad(dkb, orc, n_children):
    """Steps of ns batches in descending sample order, each sample twice in a step; qual NULL
    in one batch and present in the others; calls equal the oracle's."""
    k = 31
    if n_children == 1:
        fam = synth.make_trio_host(150_000, 15, 30, k, seed=51, indel_frac=0.3)
    else:
        fam = synth.make_family_host(150_000, 15, 30, k, n_children, seed=52, indel_frac=0.3)
    ns = 2 + n_children
    entries = dkb.variant_kmers(fam.variant_tuples(), k)
    batches = _split(dkb, fam, range(ns), 2)
    batches[1] = _noqual(dkb, batches[1])
    rev = batches[::-1]
    steps = [rev[:ns], rev[ns:]]
    assert all(len({b[0] for b in st}) < len(st) for st in steps)  # a sample twice in every step
    want, m = _check_forms(dkb, orc, entries, k, steps, ns, n_children=n_children)
    assert m["launches"] == 2
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    o_hits, o_dist, o_nk, o_calls = family_results(orc, ks, want, len(fam.variants), n_children, THR)
    hits, dist, nk, calls = m["res"]
    assert np.array_equal(hits.astype(np.uint64), o_hits) and np.array_equal(dist.astype(np.uint64), o_dist)
    assert np.array_equal(nk, o_nk)
    assert np.array_equal(calls.reshape(len(fam.variants), n_children), o_calls)


# ---- edges ----------------------------------------------------------------------------------------
def _edge_batches(dkb, k):
    """Batches of exactly n positions at +-1 of a 32-position mask word and of a 2048-position
    zero-list block; reads of length 0, k-1, k, k+1 and odd lengths; a batch whose flags are
    half unusable (plain-bits zero-list blocks); an empty batch."""
    fam = synth.make_trio_host(80_000, 30, 20, k, seed=53, n_rate=0.01)
    seq0, qual0, off0 = fam.reads[0]
    src = [(seq0[int(off0[r]):int(off0[r + 1])], qual0[int(off0[r]):int(off0[r + 1])]) for r in range(len(off0) - 1)]
    it = iter(range(len(src)))

    def batch(smp, n_pos, lens=()):
        reads, left = [], n_pos
        for L in lens:
            s, q = src[next(it)]
            reads.append((s[:L], q[:L]))
            left -= L + 1
        while left > 151:
            reads.append(src[next(it)])
            left -= len(reads[-1][0]) + 1
        if left > 0:
            s, q = src[next(it)]
            reads.append((s[:left - 1], q[:left - 1]))
        seq = np.concatenate([r[0] for r in reads]) if reads else np.zeros(0, np.uint8)
        qual = np.concatenate([r[1] for r in reads]) if reads else np.zeros(0, np.uint8)
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(r[0]) for r in reads])
        st = dkb.pack_reads(seq, qual, off, MIN_BQ)
        assert st.n_positions == n_pos
        lo = np.zeros(len(reads), np.uint64)
        return (smp, st, dkb.ReadLoci(off, lo, lo + np.uint64(1 << 40)), seq, qual, off)

    sizes = [31, 32, 33, 2047, 2048, 2049, 4095, 6145, 1, 97]
    out = [batch(i % 3, n) for i, n in enumerate(sizes)]
    out.append(batch(0, 600, [0, k - 1, k, k + 1, 1, 0, 149, 3]))
    out.append(batch(1, 3 * 2048 + 1, [0, 0, k - 1, k + 1]))
    noisy = batch(2, 5 * 2048 - 1)
    noisy[4][1::2] = 2  # every other base unusable: the zero list codes these blocks as plain bits
    noisy = (2, dkb.pack_reads(noisy[3], noisy[4], noisy[5], MIN_BQ), *noisy[2:])
    zoff, _ = dkb.mask_to_zero_list(noisy[1].mask1, noisy[1].n_positions)
    assert (zoff[:-1] & np.uint32(0x80000000)).any()
    out.append(noisy)
    empty = batch(1, 0)
    assert empty[1].n_positions == 0 and len(empty[5]) == 1
    return fam, out, empty


@pytest.mark.parametrize("form", FORMS)
def test_edges(dkb, orc, form):
    k = 31
    fam, edge, empty = _edge_batches(dkb, k)
    entries = dkb.variant_kmers(fam.variant_tuples(), k)
    edge[4] = _noqual(dkb, edge[4])
    steps = [edge[0:3] + [empty], [empty, empty], edge[3:7], [edge[7], empty, edge[8]], edge[9:12], [edge[12]]]
    assert sorted(id(b) for st in steps for b in st if b is not empty) == sorted(id(b) for b in edge)
    _check_forms(dkb, orc, entries, k, steps, 3, forms=(form,))
    with dkb.KmerCounter(k) as kc:  # n_batches 0, and a call of empty batches only: no launch
        kc.build_table(entries)
        l0 = kc.stats()["scan_launches"]
        _multi(dkb, kc, form, [])
        _multi(dkb, kc, form, [empty, empty, empty, empty])
        kc.sync()
        assert kc.stats()["scan_launches"] == l0


@pytest.mark.parametrize("regions", [False, True])
def test_adversarial_batch_edges(dkb, orc, regions):
    """tests/adversarial.py: alt windows that start and end every batch, low-complexity runs,
    batch lengths at every residue of a 16 384-position macro tile - four batches, one launch."""
    k = 31
    inp = adv.build(dkb, k, seed=k)
    entries = dkb.variant_kmers(inp.variants, k)
    batches = [(b.sample, dkb.pack_reads(b.seq, b.qual, b.off, adv.MIN_BQ), dkb.ReadLoci(b.off, b.lo, b.hi),
                b.seq, b.qual, b.off) for b in inp.batches]
    assert len(batches) == 4
    _check_forms(dkb, orc, entries, k, [batches], 3, (inp.vlo, inp.vhi) if regions else None)


# ---- region mode ------------------------------------------------------------------------------------
@pytest.mark.parametrize("tuning", TUNINGS)
@pytest.mark.parametrize("hints", [True, False])
def test_region_tunings(dkb, orc, tuning, hints):
    trio = _trimmed(synth.make_trio_host(200_000, 12, 40, 31, seed=5))
    entries = dkb.variant_kmers(trio.variant_tuples(), 31)
    batches = _split(dkb, trio, range(3), 2)
    _check_forms(dkb, orc, entries, 31, _steps(batches, 3), 3, ro.windows(trio.variants, 300),
                 tuning=tuning, hints=hints)


@pytest.mark.parametrize("k", [15, 21, 31])
def test_region_k(dkb, orc, k):
    trio = _trimmed(synth.make_trio_host(100_000, 10, 20, k, seed=7 + k))
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    batches = _split(dkb, trio, range(3), 3)
    _check_forms(dkb, orc, entries, k, _steps(batches, 3), 3, ro.windows(trio.variants, 100))


def test_region_quad(dkb, orc):
    fam = synth.make_family_host(150_000, 12, 30, 31, 2, seed=44, indel_frac=0.3)
    _trimmed(fam)
    entries = dkb.variant_kmers(fam.variant_tuples(), 31)
    batches = _split(dkb, fam, range(4), 3)
    _check_forms(dkb, orc, entries, 31, _steps(batches, 4), 4, ro.windows(fam.variants, 300),
                 n_children=2)


# ---- pipelining ------------------------------------------------------------------------------------
@pytest.mark.parametrize("regions, parts", [pytest.param(r, p, id=f"{r}{'-uneven' if p == UNEVEN else ''}")
                                            for p in (10, UNEVEN) for r in (False, True)])
def test_pipelined(dkb, orc, regions, parts):
    """New and old forms in a row without dkb_sync: sparse / reads / 4-bit multi submits, host
    multi submits and single submits of every host form; the uneven split makes each staging
    slot's seq / qual / offsets / nibble / zero-list buffers grow while the other slot's scan is
    queued.  Then the same steps with reduce_push / reduce_flush after each."""
    k = 31
    trio = _trimmed(synth.make_trio_host(200_000, 12, 30, k, seed=45))
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    vlo, vhi = ro.windows(trio.variants, 400)
    batches = _split(dkb, trio, range(3), parts)
    batches[2] = _noqual(dkb, batches[2])
    if regions:
        want = _region_want(orc, entries, batches, vlo, vhi, k, 3)
    else:
        ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
        want = np.zeros((3, len(entries)), dtype=np.uint64)
        for smp, _, _, seq, qual, off in batches:
            ks.count_reads(seq, qual, off, k, MIN_BQ, counts=want[smp])
    steps = _steps(batches, 3)
    kinds = ("sparse", "reads4", "reads", "host", "single")
    for reduce in (False, True):
        keep = []
        with dkb.KmerCounter(k) as kc:
            kc.build_table(entries)
            if regions:
                kc.set_regions(vlo, vhi)
            l0 = kc.stats()["scan_launches"]
            launches = 0
            for i, step in enumerate(steps):
                kind = kinds[i % len(kinds)]
                if kind == "single":
                    for j, b in enumerate(step):
                        _single(dkb, kc, ("sparse", "reads4", "reads")[j % 3], b, b[2] if regions else None)
                        launches += b[1].n_positions > 0
                elif kind == "host":
                    _submit_step(dkb, kc, step, "host", regions, keep)
                    launches += 1
                else:
                    _multi(dkb, kc, kind, step, [b[2] for b in step] if regions else None)
                    launches += 1
                if reduce:
                    kc.reduce_push(THR)
            if reduce:
                kc.reduce_flush(THR)
                red = kc.reduced_counts().copy()
                _, _, _, calls = kc.results()
            kc.sync()
            assert kc.stats()["scan_launches"] - l0 == launches
            got = kc.entry_counts().copy()
            assert np.array_equal(got.astype(np.uint64), want), (regions, reduce)
            if reduce:
                assert np.array_equal(red, got)
                assert np.array_equal(calls, kc.finalise(THR)[3])
    assert want.sum() > 0


# ---- refusals ---------------------------------------------------------------------------------------
def test_refusals(dkb, orc):
    from denovo_kmer_b200 import _lib
    L = _lib.lib()
    k = 31
    trio = synth.make_trio_host(20_000, 6, 4, k, seed=2)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    b = _split(dkb, trio, range(3), 1)
    three, three_loci = [x[1] for x in b], [x[2] for x in b]
    zl = [dkb.mask_to_zero_list(s.mask1, s.n_positions) for s in three]
    u64 = lambda a: np.ascontiguousarray(a, dtype=np.uint64).ctypes.data_as(_lib.u64p)  # noqa: E731
    keep = []

    def arr(t, xs, n):
        a = (t * max(n, 1))(*xs[:max(n, 0)])
        keep.append(a)
        return a

    def sparse(h, zls, smps, n=None, sts=three):
        n = len(smps) if n is None else n
        return L.dkb_batch_submit_sparse_multi(
            h, n, arr(C.c_void_p, [s.bases2.ctypes.data for s in sts], n),
            arr(C.c_void_p, [z[0].ctypes.data for z in zls], n), arr(C.c_void_p, [z[1].ctypes.data for z in zls], n),
            arr(C.c_size_t, [len(z[1]) for z in zls], n), arr(C.c_uint64, [s.n_positions for s in sts], n),
            arr(C.c_int, smps, n))

    def reads(h, offs, smps, n=None, fmt=0):
        n = len(smps) if n is None else n
        return L.dkb_batch_submit_reads_multi(
            h, n, arr(C.c_void_p, [x[3].ctypes.data for x in b], n), fmt,
            arr(C.c_void_p, [x[4].ctypes.data for x in b], n), arr(C.c_void_p, [o.ctypes.data for o in offs], n),
            arr(C.c_size_t, [len(o) - 1 for o in offs], n), MIN_BQ, arr(C.c_int, smps, n))

    def set_multi(h, ls):
        return L.dkb_batch_set_loci_multi(h, len(ls), arr(_lib.u64p, [u64(x.offsets) for x in ls], len(ls)),
                                          arr(_lib.u64p, [u64(x.lo) for x in ls], len(ls)),
                                          arr(_lib.u64p, [u64(x.hi) for x in ls], len(ls)),
                                          arr(C.c_size_t, [len(x.offsets) - 1 for x in ls], len(ls)))

    offs = [x[5] for x in b]
    desc = offs[1].copy()
    desc[3] = desc[4] + 1
    # batch 2's zero list: block offsets that do not ascend / do not end at zbytes_used
    z2 = zl[2][0].copy()
    assert len(z2) > 2
    z2[1] = z2[2] + 1
    bad_zl = [zl[0], zl[1], (z2, zl[2][1])]
    short_zl = [zl[0], zl[1], (zl[2][0].copy(), zl[2][1][:-1])]
    with dkb.KmerCounter(k) as kc:
        h = kc._h
        kc.build_table(entries)
        for fn in (lambda n: sparse(h, zl * 2, [0, 1, 2] * 2, n=n, sts=three * 2),
                   lambda n: reads(h, offs * 2, [0, 1, 2] * 2, n=n)):
            assert fn(5) == _lib.EINVAL and fn(-1) == _lib.EINVAL  # n_batches out of range
        assert sparse(h, bad_zl, [0, 1, 2]) == _lib.EINVAL
        assert b"batch 2: malformed zero list" in L.dkb_last_error(h)
        assert sparse(h, short_zl, [0, 1, 2]) == _lib.EINVAL
        assert b"batch 2: zoff[n_blocks] != zbytes_used" in L.dkb_last_error(h)
        assert sparse(h, zl, [0, 1, 3]) == _lib.EINVAL  # a bad sample
        assert reads(h, offs, [0, 1, 2], fmt=2) == _lib.EINVAL
        assert b"seq_format" in L.dkb_last_error(h)
        assert reads(h, [offs[0], desc, offs[2]], [0, 1, 2]) == _lib.EINVAL
        assert b"batch 1: offsets must not decrease" in L.dkb_last_error(h)
        assert reads(h, offs, [0, -1, 2]) == _lib.EINVAL
        assert set_multi(h, three_loci) == _lib.ESTATE  # whole-stream mode
        kc.sync()
        assert kc.stats()["scan_launches"] == 0
        kc.set_regions(*ro.windows(trio.variants, 100))
        for fn in (lambda: sparse(h, zl, [0, 1, 2]), lambda: reads(h, offs, [0, 1, 2]),
                   lambda: reads(h, offs, [0, 1, 2], fmt=1)):
            assert fn() == _lib.ESTATE  # no loci
            loci = three_loci[0]
            assert L.dkb_batch_set_loci(h, u64(loci.offsets), u64(loci.lo), u64(loci.hi),
                                        len(loci.offsets) - 1) == _lib.OK
            assert fn() == _lib.ESTATE  # single-batch loci pending
            assert fn() == _lib.ESTATE  # used up
            assert set_multi(h, three_loci[:2]) == _lib.OK
            assert fn() == _lib.EINVAL  # loci for two batches, three submitted
            short = dkb.ReadLoci(loci.offsets[:-1], loci.lo[:-1], loci.hi[:-1])
            assert set_multi(h, [short] + three_loci[1:]) == _lib.OK
            assert fn() == _lib.EINVAL  # batch 0's loci cover other positions
            assert b"batch 0: " in L.dkb_last_error(h)
            assert fn() == _lib.ESTATE  # used up by the refusal
        # refusals of the batches themselves use up the loci too (EINVAL before ESTATE)
        assert set_multi(h, three_loci) == _lib.OK
        assert sparse(h, bad_zl, [0, 1, 2]) == _lib.EINVAL
        assert sparse(h, zl, [0, 1, 2]) == _lib.ESTATE
        assert set_multi(h, three_loci) == _lib.OK
        assert reads(h, [offs[0], desc, offs[2]], [0, 1, 2]) == _lib.EINVAL
        assert reads(h, offs, [0, 1, 2]) == _lib.ESTATE
        # profiling counters: refused in region mode
        kc.profile_counters(True)
        assert set_multi(h, three_loci) == _lib.OK
        assert sparse(h, zl, [0, 1, 2]) == _lib.ESTATE
        assert set_multi(h, three_loci) == _lib.OK
        assert reads(h, offs, [0, 1, 2]) == _lib.ESTATE
        kc.profile_counters(False)
        kc.sync()
        assert kc.stats()["scan_launches"] == 0
        # and correct submits afterwards count right: one launch each
        kc.reset_counts()
        _multi(dkb, kc, "sparse", b, three_loci)
        _multi(dkb, kc, "reads", b, three_loci)
        _multi(dkb, kc, "reads4", b, three_loci)
        kc.sync()
        assert kc.stats()["scan_launches"] == 3
        got = kc.entry_counts().copy()
    vlo, vhi = ro.windows(trio.variants, 100)
    want = _region_want(orc, entries, b, vlo, vhi, k, 3)
    assert np.array_equal(got.astype(np.uint64), 3 * want) and want.sum() > 0
