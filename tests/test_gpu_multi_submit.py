"""-m gpu: multi-batch submits - dkb_batch_submit_multi (host memory) and, in region mode,
dkb_batch_submit_multi / dkb_batch_submit_device_multi with dkb_batch_set_loci_multi - scan up
to four batches in one launch and count exactly what one submit per batch counts: the oracle
(whole stream) and the region oracle (tests/region_oracle.c) bit for bit, over tunings, k,
indels, families, uneven segments, the edges of the per-segment locus index, every region twin
of the scan kernel with several segments, pipelined submits, and every refusal."""
import ctypes as C
import itertools

import numpy as np
import pytest

import adversarial as adv
import region_oracle as ro
from denovo_kmer_b200 import synth
from family_oracle import family_results
from helpers import oracle_counts
from test_gpu_regions import TUNINGS, _submit, _trimmed

pytestmark = pytest.mark.gpu

THR = (3, 2, 0, 1)
MIN_BQ = 20


def _split(dkb, fam, samples, parts, min_bq=MIN_BQ):
    """Per sample, its reads cut into `parts` batches - that many even ones, or a list of the
    batches' relative sizes: [(sample, stream, loci, seq, qual, off)]."""
    out = []
    for smp in samples:
        seq, qual, off = fam.reads[smp]
        lo, hi = fam.loci[smp]
        if np.isscalar(parts):
            cuts = np.linspace(0, len(off) - 1, parts + 1).astype(int)
        else:
            cuts = (np.cumsum([0] + list(parts)) / sum(parts) * (len(off) - 1)).astype(int)
        for a, b in zip(cuts[:-1], cuts[1:]):
            a0, b0 = int(off[a]), int(off[b])
            boff = off[a:b + 1] - off[a]
            out.append((smp, dkb.pack_reads(seq[a0:b0], qual[a0:b0], boff, min_bq),
                        dkb.ReadLoci(boff, lo[a:b], hi[a:b]), seq[a0:b0], qual[a0:b0], boff))
    return out


def _region_want(orc, entries, batches, vlo, vhi, k, ns, min_bq=MIN_BQ):
    want = np.zeros((ns, len(entries)), dtype=np.uint64)
    for smp, _, loci, seq, qual, off in batches:
        if len(off) < 2:
            continue
        b2, m1, n_pos = orc.pack_stream(seq, qual, off, min_bq)
        ro.count_stream_loci(entries.keys, entries.variant, entries.allele, vlo, vhi, b2, m1, n_pos, off, loci.lo,
                             loci.hi, k, counts=want[smp])
    return want


def _steps(batches, width):
    """Group batches into launches of up to `width`, taking them round-robin over the samples so
    that a launch mixes samples."""
    by = {}
    for b in batches:
        by.setdefault(b[0], []).append(b)
    order = [b for grp in itertools.zip_longest(*by.values()) for b in grp if b is not None]
    return [order[i:i + width] for i in range(0, len(order), width)]


def _device(dkb, stream):
    import torch
    return (torch.from_numpy(stream.bases2.view(np.int32).copy()).cuda(),
            torch.from_numpy(stream.mask1.view(np.int32).copy()).cuda())


def _submit_step(dkb, kc, step, form, regions, keep):
    loci = [b[2] for b in step] if regions else None
    if form == "host":
        kc.submit_multi([b[1] for b in step], [b[0] for b in step], loci=loci)
    else:
        dev = [_device(dkb, b[1]) for b in step]
        keep.append(dev)  # alive until the sync below
        kc.submit_device_multi([(d[0].data_ptr(), d[1].data_ptr(), b[1].n_positions, b[0]) for d, b in zip(dev, step)],
                               loci=loci)


def _run(dkb, entries, k, steps, form="host", vlo=None, vhi=None, tuning=None, hints=True, n_children=1):
    keep = []
    with dkb.KmerCounter(k, tuning=tuning, n_children=n_children) as kc:
        kc.build_table(entries, use_window_hints=hints)
        if vlo is not None:
            kc.set_regions(vlo, vhi)
        l0 = kc.stats()["scan_launches"]
        for step in steps:
            _submit_step(dkb, kc, step, form, vlo is not None, keep)
        kc.sync()
        keep.clear()
        st = kc.stats()
        got = kc.entry_counts().copy()
        res = kc.finalise(THR)
        tun = kc.tuning()
    return got, res, tun, st["scan_launches"] - l0, st


def _region_check(dkb, orc, fam, k, pad=500, form="host", parts=2, n_children=1, drop_shared=True, **kw):
    entries = dkb.variant_kmers(fam.variant_tuples(), k, drop_shared=drop_shared)
    vlo, vhi = ro.windows(fam.variants, pad)
    ns = 2 + n_children
    batches = _split(dkb, fam, range(ns), parts)
    want = _region_want(orc, entries, batches, vlo, vhi, k, ns)
    got, _, tun, launches, _ = _run(dkb, entries, k, _steps(batches, 4 if ns > 3 else 3), form, vlo, vhi,
                                    n_children=n_children, **kw)
    bad = np.argwhere(got.astype(np.uint64) != want)
    assert len(bad) == 0, (tun, form, len(bad), [(int(s), int(e), int(got[s, e]), int(want[s, e])) for s, e in bad[:5]])
    assert want.sum() > 0
    assert launches == len(_steps(batches, 4 if ns > 3 else 3))
    return want


# ---- whole-stream host multi ----------------------------------------------------------
@pytest.mark.parametrize("n_children", [1, 2])
def test_host_multi_whole_stream(dkb, orc, n_children):
    """A trio (three batches per launch) and a quad (four): counters, statistics and calls equal
    the oracle and one submit per batch; one scan launch per multi submit."""
    k = 31
    if n_children == 1:
        fam = synth.make_trio_host(150_000, 15, 30, k, seed=41, indel_frac=0.3)
    else:
        fam = synth.make_family_host(150_000, 15, 30, k, n_children, seed=42, indel_frac=0.3)
    ns = 2 + n_children
    entries = dkb.variant_kmers(fam.variant_tuples(), k)
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    want = np.zeros((ns, len(entries)), dtype=np.uint64)
    for smp in range(ns):
        ks.count_reads(*fam.reads[smp], k, MIN_BQ, counts=want[smp])
    batches = _split(dkb, fam, range(ns), 2)
    steps = _steps(batches, ns)
    got, (hits, dist, nk, calls), _, launches, _ = _run(dkb, entries, k, steps, n_children=n_children)
    assert np.array_equal(got.astype(np.uint64), want) and want.sum() > 0
    assert launches == len(steps) == 2
    o_hits, o_dist, o_nk, o_calls = family_results(orc, ks, want, len(fam.variants), n_children, THR)
    assert np.array_equal(hits.astype(np.uint64), o_hits) and np.array_equal(dist.astype(np.uint64), o_dist)
    assert np.array_equal(nk, o_nk)
    assert np.array_equal(calls.reshape(len(fam.variants), n_children), o_calls)
    # the same batches one submit each
    with dkb.KmerCounter(k, n_children=n_children) as kc:
        kc.build_table(entries)
        for smp, st, *_ in batches:
            kc.submit(st, smp)
        assert np.array_equal(kc.entry_counts(), got)
        assert np.array_equal(kc.finalise(THR)[3], calls)


def test_host_multi_order_repeats_and_empty(dkb, orc):
    """Batches in any sample order, one sample twice in a launch, batches of 0 positions, and
    n_batches = 0; only launches with positions count as scan launches."""
    k = 31
    trio = synth.make_trio_host(100_000, 12, 20, k, seed=43)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    _, want = oracle_counts(orc, entries, trio, k, MIN_BQ)
    b = _split(dkb, trio, range(3), 2)  # (s0a, s0b, s1a, s1b, s2a, s2b)
    empty = dkb.pack_reads(np.zeros(0, np.uint8), np.zeros(0, np.uint8), np.zeros(1, np.uint64), MIN_BQ)
    assert empty.n_positions == 0
    with dkb.KmerCounter(k) as kc:
        kc.build_table(entries)
        l0 = kc.stats()["scan_launches"]
        kc.submit_multi([], [])
        kc.submit_multi([empty, empty], [2, 0])
        assert kc.stats()["scan_launches"] == l0
        kc.submit_multi([b[5][1], b[0][1], b[1][1], empty], [2, 0, 0, 1])  # sample 0 twice, reversed order
        kc.submit_multi([b[3][1], b[2][1], b[4][1]], [1, 1, 2])
        assert kc.stats()["scan_launches"] == l0 + 2
        assert np.array_equal(kc.entry_counts().astype(np.uint64), want) and want.sum() > 0


# ---- region mode ---------------------------------------------------------------------------
@pytest.mark.parametrize("tuning", TUNINGS)
@pytest.mark.parametrize("hints", [True, False])
def test_region_multi_tunings(dkb, orc, tuning, hints):
    trio = _trimmed(synth.make_trio_host(200_000, 12, 40, 31, seed=5))
    for form in ("host", "device"):
        _region_check(dkb, orc, trio, 31, pad=300, form=form, tuning=tuning, hints=hints)


@pytest.mark.parametrize("gate", ["0", "1"])
@pytest.mark.parametrize("tuning", [(15, 16, 2, 2), (13, 8, 1, 2), (9, 16, 2, 2)])
def test_region_multi_gated_lookups(dkb, orc, tuning, gate, monkeypatch):
    monkeypatch.setenv("DKB_GATE", gate)
    trio = _trimmed(synth.make_trio_host(150_000, 14, 30, 31, seed=77, n_rate=0.01, lowq_frac=0.08, ragged=True))
    _region_check(dkb, orc, trio, 31, tuning=tuning, parts=3)


@pytest.mark.parametrize("k", [15, 21, 31])
def test_region_multi_k(dkb, orc, k):
    trio = _trimmed(synth.make_trio_host(100_000, 10, 20, k, seed=7 + k))
    _region_check(dkb, orc, trio, k, pad=100)
    _region_check(dkb, orc, trio, k, pad=100, form="device", hints=False, tuning=(0, 2, 0))


@pytest.mark.parametrize("drop_shared", [True, False])
def test_region_multi_indels(dkb, orc, drop_shared):
    trio = _trimmed(synth.make_trio_host(150_000, 15, 40, 31, seed=11, indel_frac=0.6))
    _region_check(dkb, orc, trio, 31, pad=50, drop_shared=drop_shared)


@pytest.mark.parametrize("form", ["host", "device"])
def test_region_multi_quad(dkb, orc, form):
    fam = synth.make_family_host(150_000, 12, 30, 31, 2, seed=44, indel_frac=0.3)
    _trimmed(fam)  # (moves reads of samples 0..2; sample 3 keeps its loci)
    _region_check(dkb, orc, fam, 31, pad=300, form=form, n_children=2, parts=3)


def _edge_batch(k, seed=4):
    """Reads crossing 2048-position tiles, reads longer than a tile, empty and unmapped reads."""
    rng = np.random.default_rng(seed)
    genome = synth.make_genome(60_000, 8)
    variants = synth.plant_variants(genome, 12, k, 9)
    alt = synth.apply_variants(genome, variants)
    rp = synth.hap_ref_positions(genome, variants)
    lens = [5000, 0, 150, 3000, 0, 2100, 2048, 31, 4000, 1, 150] * 4
    seqs, lo, hi = [], [], []
    for n in lens:
        s = int(rng.integers(0, len(alt) - max(n, 1)))
        seqs.append(alt[s:s + n])
        lo.append(int(rp[s]))
        hi.append(int(rp[s + n - 1]) + 1 if n else int(rp[s]))
    seq = np.concatenate(seqs)
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(x) for x in seqs])
    lo, hi = np.array(lo, np.uint64), np.array(hi, np.uint64)
    hi[3::7] = lo[3::7]  # unmapped
    return genome, variants, seq, np.full(len(seq), 30, np.uint8), off, lo, hi


@pytest.mark.parametrize("tuning", [None, (15, 2, 2), (15, 16, 2, 2), (12, 1, 1), (14, 4, 1, 2)])
@pytest.mark.parametrize("form", ["host", "device"])
def test_region_multi_uneven_segments_and_edges(dkb, orc, tuning, form):
    """One launch holds: a batch of three reads (fewer work units than warps), the edge batch
    (tile-crossing, long, empty and unmapped reads), a batch none of whose reads overlaps any
    window, and a full batch; then the same batches in another order."""
    k = 31
    genome, variants, seq, qual, off, lo, hi = _edge_batch(k)
    fam = synth.Trio(k, genome, variants)
    full = synth.make_trio_host(60_000, 20, 1, k, seed=8)  # same genome (seed 8), its own reads
    fseq, fqual, foff = full.reads[1]
    flo, fhi = full.loci[1]
    fam.reads = {0: (seq, qual, off), 1: (fseq, fqual, foff), 2: (fseq[:450], fqual[:450], foff[:4])}
    fam.loci = {0: (lo, hi), 1: (flo, fhi), 2: (flo[:3], fhi[:3])}
    batches = _split(dkb, fam, range(3), 1)
    # a far-away copy of the full batch: no read overlaps a window
    far = dkb.ReadLoci(batches[1][2].offsets, batches[1][2].lo + np.uint64(1 << 40), batches[1][2].hi + np.uint64(1 << 40))
    batches.append((2, batches[1][1], far, *batches[1][3:]))
    entries = dkb.variant_kmers(fam.variant_tuples(), k)
    vlo, vhi = ro.windows(variants, 2000)
    vhi[2] = vlo[2]  # an empty window
    want = _region_want(orc, entries, batches, vlo, vhi, k, 3)
    assert want[0].sum() > 0 and want[1].sum() > 0
    order = [batches[2], batches[0], batches[3], batches[1]]
    for steps in ([order], [batches[::-1]], [batches[:3], batches[3:]]):
        got, _, tun, launches, _ = _run(dkb, entries, k, steps, form, vlo, vhi, tuning=tuning)
        assert np.array_equal(got.astype(np.uint64), want), (tun, form, len(steps))
        assert launches == len(steps)


# ---- every region twin with several segments -------------------------------------------------
STRIDES, HASHES = (1, 2, 4, 8, 16), (1, 2, 3, 4)
MODES = {"smem": (1, None), "l2": (2, "0"), "l2_pre": (2, "37120")}  # filter_mode, DKB_PREFILTER_WORDS


@pytest.fixture(scope="module")
def adv_input(dkb, orc):
    k = 31
    inp = adv.build(dkb, k, seed=k)
    entries = dkb.variant_kmers(inp.variants, k)
    batches = [(b.sample, dkb.pack_reads(b.seq, b.qual, b.off, adv.MIN_BQ), dkb.ReadLoci(b.off, b.lo, b.hi),
                b.seq, b.qual, b.off) for b in inp.batches]
    assert len(batches) >= 3
    want = _region_want(orc, entries, batches, inp.vlo, inp.vhi, k, 3, adv.MIN_BQ)
    assert want.sum() > 0
    return dict(inp=inp, entries=entries, batches=batches, want=want)


def test_every_region_twin_with_several_segments(dkb, adv_input, monkeypatch):
    """Each of the 44 region twins of k_scan, forced by tuning, DKB_PREFILTER_WORDS and DKB_GATE,
    scans the adversarial trio's four batches in ONE launch (host and device forms alternate)."""
    d = adv_input
    inp, seen, failures = d["inp"], set(), []
    for i, (D, NH, mode, gate) in enumerate(itertools.product(STRIDES, HASHES, MODES, (False, True))):
        fmode, pre = MODES[mode]
        if mode != "smem" and (D == 1 or NH > 2):
            continue  # not built
        fm = 0 if mode == "smem" else (2 if mode == "l2_pre" else 1) + (2 if gate and D >= 8 else 0)
        if (D, NH, fm) in seen:
            continue  # the gate is ignored here: same kernel
        if pre is None:
            monkeypatch.delenv("DKB_PREFILTER_WORDS", raising=False)
        else:
            monkeypatch.setenv("DKB_PREFILTER_WORDS", pre)
        monkeypatch.setenv("DKB_GATE", "1" if gate else "0")
        s = min(15, 31 - D + 1)
        form = "host" if len(seen) % 2 == 0 else "device"
        got, _, tun, launches, st = _run(dkb, d["entries"], 31, [d["batches"]], form, inp.vlo, inp.vhi,
                                         tuning=(s, D, NH, fmode))
        assert tun == (s, D, NH, fmode)
        assert (st["prefilter_words"] > 0) == (fm in (2, 4)) and st["gated_lookups"] == (fm >= 3)
        assert launches == 1
        bad = np.argwhere(got.astype(np.uint64) != d["want"])
        if len(bad):
            failures.append(f"region twin {(D, NH, fm)} ({form}): {len(bad)} counters differ")
        seen.add((D, NH, fm))
    assert not failures, "\n".join(failures)
    assert len(seen) == 44


# ---- pipelining ----------------------------------------------------------------------------
SINGLE_FORMS = ("submit", "sparse", "reads", "reads4")
UNEVEN = (1, 6, 1, 10, 10, 10, 1, 6)


@pytest.mark.parametrize("regions, parts", [pytest.param(r, p, id=f"{r}{'-uneven' if p == UNEVEN else ''}")
                                            for p in (10, UNEVEN) for r in (False, True)])
def test_multi_pipelined(dkb, orc, regions, parts):
    """Multi submits in a row without dkb_sync, interleaved with single submits (host and
    device multi; dkb_batch_submit, _sparse, _reads from ASCII and from 4-bit codes), so that
    every form shares both staging buffers and both locus stages; then the same steps with
    reduce_push / reduce_flush after each on one GPU.  The uneven split makes each staging
    buffer and each locus stage grow while the other one's scan is queued."""
    k = 31
    trio = _trimmed(synth.make_trio_host(200_000, 12, 30, k, seed=45))
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    vlo, vhi = ro.windows(trio.variants, 400)
    batches = _split(dkb, trio, range(3), parts)
    if regions:
        want = _region_want(orc, entries, batches, vlo, vhi, k, 3)
    else:
        ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
        want = np.zeros((3, len(entries)), dtype=np.uint64)
        for smp in range(3):
            ks.count_reads(*trio.reads[smp], k, MIN_BQ, counts=want[smp])
    steps = _steps(batches, 3)
    assert len(steps) == (parts if np.isscalar(parts) else len(parts))
    for reduce in (False, True):
        keep = []
        with dkb.KmerCounter(k) as kc:
            kc.build_table(entries)
            if regions:
                kc.set_regions(vlo, vhi)
            l0 = kc.stats()["scan_launches"]
            n_multi = n_single = launches = 0
            for i, step in enumerate(steps):
                if i % 4 == 3:  # a single-batch submit per batch of this step, the forms in turn
                    for smp, st, loci, seq, qual, off in step:
                        _submit(dkb, kc, SINGLE_FORMS[n_single % 4], seq, qual, off, smp, MIN_BQ,
                                loci if regions else None)
                        n_single += 1
                        launches += st.n_positions > 0
                else:
                    _submit_step(dkb, kc, step, "device" if i % 4 == 2 else "host", regions, keep)
                    n_multi += 1
                    launches += any(b[1].n_positions > 0 for b in step)
                if reduce:
                    kc.reduce_push(THR)
            assert n_multi >= 6 and n_single >= len(SINGLE_FORMS)
            if reduce:
                kc.reduce_flush(THR)
                red = kc.reduced_counts().copy()
                _, _, _, calls = kc.results()
            kc.sync()
            keep.clear()
            assert kc.stats()["scan_launches"] - l0 == launches
            got = kc.entry_counts().copy()
            assert np.array_equal(got.astype(np.uint64), want), (regions, reduce)
            if reduce:
                assert np.array_equal(red, got)
                assert np.array_equal(calls, kc.finalise(THR)[3])
    assert want.sum() > 0


# ---- refusals ------------------------------------------------------------------------------
def test_multi_refusals(dkb):
    from denovo_kmer_b200 import _lib
    L = _lib.lib()
    k = 31
    trio = synth.make_trio_host(20_000, 6, 4, k, seed=2)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    b = _split(dkb, trio, range(3), 1)
    st, loci = b[0][1], b[0][2]
    u64 = lambda a: np.ascontiguousarray(a, dtype=np.uint64).ctypes.data_as(_lib.u64p)  # noqa: E731
    keep = []

    def set_multi(h, ls, n=None, n_reads=None):
        n = len(ls) if n is None else n
        m = max(n, 0)
        arr = lambda f: (_lib.u64p * max(n, 1))(*[u64(getattr(x, f)) for x in ls][:m])  # noqa: E731
        nr = (C.c_size_t * max(n, 1))(*(n_reads or [len(x.offsets) - 1 for x in ls])[:m])
        keep.append((ls, arr, nr))
        return L.dkb_batch_set_loci_multi(h, n, arr("offsets"), arr("lo"), arr("hi"), nr)

    def submit(h, sts, smps, n=None):
        n = len(sts) if n is None else n
        m = max(n, 0)
        bb = (C.c_void_p * max(n, 1))(*[s.bases2.ctypes.data for s in sts][:m])
        mm = (C.c_void_p * max(n, 1))(*[s.mask1.ctypes.data for s in sts][:m])
        npos = (C.c_uint64 * max(n, 1))(*[s.n_positions for s in sts][:m])
        smp = (C.c_int * max(n, 1))(*smps[:m])
        return L.dkb_batch_submit_multi(h, n, bb, mm, npos, smp)

    three = [x[1] for x in b]
    three_loci = [x[2] for x in b]
    with dkb.KmerCounter(k) as kc:
        h = kc._h
        kc.build_table(entries)
        assert set_multi(h, three_loci) == _lib.ESTATE  # whole-stream mode
        assert submit(h, three, [0, 1, 2, 3]) == _lib.OK  # no loci needed there
        assert submit(h, three, [0, 1, 3]) == _lib.EINVAL  # a bad sample
        assert submit(h, three * 2, [0, 1, 2] * 2, n=5) == _lib.EINVAL  # n_batches out of range
        assert submit(h, three, [0, 1, 2], n=-1) == _lib.EINVAL
        kc.set_regions(*ro.windows(trio.variants, 100))
        assert submit(h, three, [0, 1, 2]) == _lib.ESTATE  # no loci
        assert submit(h, [], [], n=0) == _lib.ESTATE  # (as a single submit of 0 positions is)
        # single-batch loci before a multi submit, multi loci before a single submit
        assert L.dkb_batch_set_loci(h, u64(loci.offsets), u64(loci.lo), u64(loci.hi), len(loci.offsets) - 1) == _lib.OK
        assert submit(h, three, [0, 1, 2]) == _lib.ESTATE
        assert submit(h, three, [0, 1, 2]) == _lib.ESTATE  # used up: now none is pending
        assert set_multi(h, [loci]) == _lib.OK
        assert L.dkb_batch_submit(h, st.bases2.ctypes.data, st.mask1.ctypes.data, st.n_positions, 0) == _lib.ESTATE
        assert L.dkb_batch_submit(h, st.bases2.ctypes.data, st.mask1.ctypes.data, st.n_positions, 0) == _lib.ESTATE
        # mismatched n_batches; a batch whose loci cover other positions
        assert set_multi(h, three_loci) == _lib.OK
        assert submit(h, three[:2], [0, 1]) == _lib.EINVAL
        short = dkb.ReadLoci(loci.offsets[:-1], loci.lo[:-1], loci.hi[:-1])
        assert set_multi(h, [short] + three_loci[1:]) == _lib.OK
        assert submit(h, three, [0, 1, 2]) == _lib.EINVAL
        # the loci themselves: descending offsets, n_reads >= 2^32, n_batches out of range
        bad = loci.offsets.copy()
        bad[3] = bad[4] + 1
        assert set_multi(h, [three_loci[1], dkb.ReadLoci(bad, loci.lo, loci.hi)]) == _lib.EINVAL
        assert submit(h, three[1:], [1, 0]) == _lib.ESTATE  # nothing pending after a refused set
        assert set_multi(h, three_loci[:1], n_reads=[1 << 32]) == _lib.EINVAL
        assert set_multi(h, three_loci * 2, n=5) == _lib.EINVAL
        assert set_multi(h, three_loci, n=-1) == _lib.EINVAL
        # a bad sample, with correct loci: refused, loci used up
        assert set_multi(h, three_loci) == _lib.OK
        assert submit(h, three, [0, 1, 8]) == _lib.EINVAL
        assert submit(h, three, [0, 1, 2]) == _lib.ESTATE
        # device multi: the same rules
        import torch
        dev = [_device(dkb, s) for s in three]
        bb = (C.c_void_p * 3)(*[d[0].data_ptr() for d in dev])
        mm = (C.c_void_p * 3)(*[d[1].data_ptr() for d in dev])
        npos = (C.c_uint64 * 3)(*[s.n_positions for s in three])
        smp = (C.c_int * 3)(0, 1, 2)
        assert L.dkb_batch_submit_device_multi(h, 3, bb, mm, npos, smp) == _lib.ESTATE
        assert set_multi(h, three_loci[:2]) == _lib.OK
        assert L.dkb_batch_submit_device_multi(h, 3, bb, mm, npos, smp) == _lib.EINVAL
        # profiling on
        kc.profile_counters(True)
        assert set_multi(h, three_loci) == _lib.OK
        assert submit(h, three, [0, 1, 2]) == _lib.ESTATE
        assert set_multi(h, three_loci) == _lib.OK
        assert L.dkb_batch_submit_device_multi(h, 3, bb, mm, npos, smp) == _lib.ESTATE
        kc.profile_counters(False)
        # and correct submits afterwards count right
        kc.reset_counts()
        kc.submit_multi(three, [0, 1, 2], loci=three_loci)
        kc.submit_device_multi([(d[0].data_ptr(), d[1].data_ptr(), s.n_positions, i)
                                for i, (d, s) in enumerate(zip(dev, three))], loci=three_loci)
        kc.sync()
        got = kc.entry_counts().copy()
        torch.cuda.synchronize()
    vlo, vhi = ro.windows(trio.variants, 100)
    import oracle
    want = _region_want(oracle, entries, b, vlo, vhi, k, 3)
    assert np.array_equal(got.astype(np.uint64), 2 * want) and want.sum() > 0
