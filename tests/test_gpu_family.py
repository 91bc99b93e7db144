"""-m gpu: family contexts (one mother, one father, several children against one table) on the
B200 against the family oracle (tests/family_oracle.py, composed from the trio oracle), bit for
bit: every sample's counters, hits, distinct, n_kmers and every child's calls, over the filter
modes, every submit form, the multi-stream launch, region mode, finalise_from, the overlapped
reduction, the refusals, a full-size quad with an analytic truth, and two NCCL ranks."""
import ctypes as C
import os
import sys
import time

import numpy as np
import pytest
import torch

import region_oracle as ro
from denovo_kmer_b200 import synth
from family_oracle import family_counts, family_results

pytestmark = pytest.mark.gpu

K, THR, MIN_BQ = 31, (3, 2, 0, 1), 20
BAM_CODES = {c: i for i, c in enumerate(b"=ACMGRSVTWYHKDBN")}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _family(n_children, seed, glen=100_000, depth=10, n_var=30, **kw):
    return synth.make_family_host(glen, depth, n_var, K, n_children, seed=seed, indel_frac=0.3,
                                  shared_frac=0.3, inherited_frac=0.2, **kw)


def _oracle(dkb, orc, fam):
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    ks, counts = family_counts(orc, entries, fam, K, MIN_BQ, 2 + fam.n_children)
    return entries, counts, family_results(orc, ks, counts, len(fam.variants), fam.n_children, THR)


def _four_bit(seq, off):
    """ASCII reads -> BAM 4-bit codes, every read on a byte boundary, reads back to back."""
    out = []
    for r in range(len(off) - 1):
        s = seq[int(off[r]):int(off[r + 1])].tobytes()
        codes = [BAM_CODES.get(c, 15) for c in s.upper()] + ([0] if len(s) % 2 else [])
        out += [codes[i] << 4 | codes[i + 1] for i in range(0, len(codes), 2)]
    return np.array(out, dtype=np.uint8)


def _submit(dkb, kc, form, reads, smp, loci=None):
    seq, qual, off = reads
    if form == "reads":
        kc.submit_reads(seq, qual, off, smp, MIN_BQ, loci=loci)
        return
    if form == "reads4":
        kc.submit_reads(_four_bit(seq, off), qual, off, smp, MIN_BQ, four_bit=True, loci=loci)
        return
    st = dkb.pack_reads(seq, qual, off, MIN_BQ)
    if form == "submit":
        kc.submit(st, smp, loci=loci)
    elif form == "sparse":
        zoff, zbytes = dkb.mask_to_zero_list(st.mask1, st.n_positions)
        kc.submit_sparse(st.bases2, zoff, zbytes, st.n_positions, smp, loci=loci)
    elif form == "device":
        b2 = torch.from_numpy(st.bases2.view(np.int32).copy()).cuda()
        m1 = torch.from_numpy(st.mask1.view(np.int32).copy()).cuda()
        kc.submit_device(b2.data_ptr(), m1.data_ptr(), st.n_positions, smp, loci=loci)
        kc.sync()  # the tensors go out of scope here
    else:
        raise ValueError(form)


def _run(dkb, fam, entries, tuning=None, form="submit"):
    with dkb.KmerCounter(K, tuning=tuning, n_children=fam.n_children) as kc:
        kc.build_table(entries)
        for smp in range(kc.n_samples):
            _submit(dkb, kc, form, fam.reads[smp], smp)
        got = kc.entry_counts().copy()
        res = tuple(x.copy() for x in kc.finalise(THR))
    return got, res


def _assert_equal(got, res, want, wres):
    assert np.array_equal(got.astype(np.uint64), want), int((got != want).sum())
    hits, dist, nk, calls = res
    o_hits, o_dist, o_nk, o_calls = wres
    assert np.array_equal(hits.astype(np.uint64), o_hits) and np.array_equal(dist.astype(np.uint64), o_dist)
    assert np.array_equal(nk, o_nk)
    assert np.array_equal(calls, o_calls if o_calls.shape[1] > 1 else o_calls[:, 0])
    assert want.sum() > 0


@pytest.mark.parametrize("mode", ["smem", "l2", "l2_pre"])
@pytest.mark.parametrize("n_children", [2, 3, 6])
def test_family_parity(dkb, orc, n_children, mode, monkeypatch):
    tuning = {"smem": (0, 0, 0, 1), "l2": (15, 16, 2, 2), "l2_pre": (15, 16, 2, 2)}[mode]
    if mode != "smem":
        monkeypatch.setenv("DKB_PREFILTER_WORDS", "37120" if mode == "l2_pre" else "0")
    fam = _family(n_children, seed=100 + n_children)
    entries, want, wres = _oracle(dkb, orc, fam)
    got, res = _run(dkb, fam, entries, tuning=tuning)
    assert got.shape == (2 + n_children, len(entries)) and res[3].shape == (len(fam.variants), n_children)
    _assert_equal(got, res, want, wres)
    assert (wres[3] & 1).any(axis=0).all(), "every child has a de novo call"


def _plain_trio(dkb):
    """A KmerCounter whose context comes from dkb_ctx_create, not dkb_ctx_create_family."""
    from denovo_kmer_b200 import _lib
    kc = dkb.KmerCounter(K)
    kc._L.dkb_ctx_destroy(kc._h)
    kc._h = C.c_void_p()
    _lib.check(kc._L.dkb_ctx_create(0, K, C.byref(kc._h)))
    return kc


def test_one_child_family_is_a_trio(dkb, orc):
    trio = synth.make_trio_host(100_000, 12, 30, K, seed=8, indel_frac=0.3)
    entries = dkb.variant_kmers(trio.variant_tuples(), K)
    out = []
    for make in (lambda: _plain_trio(dkb), lambda: dkb.KmerCounter(K, n_children=1)):
        with make() as kc:
            n = C.c_int(0)
            kc._ck(kc._L.dkb_ctx_get_children(kc._h, C.byref(n)))
            assert n.value == 1 and kc.n_samples == 3
            kc.build_table(entries)
            for smp in range(3):
                kc.submit(dkb.pack_reads(*trio.reads[smp], MIN_BQ), smp)
            out.append((kc.entry_counts().copy(),) + tuple(x.copy() for x in kc.finalise(THR)))
    for a, b in zip(*out):
        assert a.shape == b.shape and np.array_equal(a, b)
    assert out[1][4].shape == (len(trio.variants),) and out[0][0].sum() > 0


def test_quad_equals_one_trio_per_child(dkb):
    fam = _family(2, seed=5)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    got, (hits, dist, nk, calls) = _run(dkb, fam, entries)
    for c in range(2):
        rows = [synth.child_sample(c), 1, 2]
        with dkb.KmerCounter(K) as kc:
            kc.build_table(entries)
            for smp, src in enumerate(rows):
                kc.submit(dkb.pack_reads(*fam.reads[src], MIN_BQ), smp)
            t_counts = kc.entry_counts()
            t_hits, t_dist, t_nk, t_calls = kc.finalise(THR)
        assert np.array_equal(got[rows], t_counts)
        assert np.array_equal(hits[:, :, rows], t_hits) and np.array_equal(dist[:, :, rows], t_dist)
        assert np.array_equal(nk, t_nk) and np.array_equal(calls[:, c], t_calls)


@pytest.mark.parametrize("form", ["submit", "sparse", "reads", "reads4", "device"])
def test_family_every_submit_form(dkb, orc, form):
    """Every single-batch submit form, with sample indices 3 and up."""
    fam = _family(3, seed=60, ragged=True, n_rate=0.01, lowq_frac=0.05)
    entries, want, wres = _oracle(dkb, orc, fam)
    got, res = _run(dkb, fam, entries, form=form)
    _assert_equal(got, res, want, wres)
    assert want[3:].sum() > 0


def test_family_multi_launch(dkb, orc):
    """A quad's four device-resident streams in one dkb_batch_submit_device_multi launch equal
    four single submits, and cost one scan launch."""
    fam = _family(2, seed=61)
    entries, want, wres = _oracle(dkb, orc, fam)
    streams = []
    for smp in range(4):
        st = dkb.pack_reads(*fam.reads[smp], MIN_BQ)
        streams.append((torch.from_numpy(st.bases2.view(np.int32).copy()).cuda(),
                        torch.from_numpy(st.mask1.view(np.int32).copy()).cuda(), st.n_positions))
    torch.cuda.synchronize()
    out = []
    for multi in (True, False):
        with dkb.KmerCounter(K, n_children=2) as kc:
            kc.build_table(entries)
            before = kc.stats()["scan_launches"]
            batches = [(b.data_ptr(), m.data_ptr(), n, smp) for smp, (b, m, n) in enumerate(streams)]
            if multi:
                kc.submit_device_multi(batches[::-1])
            else:
                for bt in batches:
                    kc.submit_device(*bt)
            launches = kc.stats()["scan_launches"] - before
            out.append((kc.entry_counts().copy(), tuple(x.copy() for x in kc.finalise(THR))))
        assert launches == (1 if multi else 4)
    assert np.array_equal(out[0][0], out[1][0])
    _assert_equal(*out[0], want, wres)


def test_family_region_mode(dkb, orc):
    fam = _family(3, seed=62, paralog_frac=0.3)
    rng = np.random.default_rng(1)
    for smp in fam.loci:  # move a third of the reads far away so that the windows cut
        lo, hi = fam.loci[smp]
        far = rng.random(len(lo)) < 0.3
        lo[far] += np.uint64(1 << 30)
        hi[far] += np.uint64(1 << 30)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    vlo, vhi = ro.windows(fam.variants, 400)
    ns = 5
    want = np.zeros((ns, len(entries)), dtype=np.uint64)
    for smp in range(ns):
        seq, qual, off = fam.reads[smp]
        b2, m1, n_pos = orc.pack_stream(seq, qual, off, MIN_BQ)
        lo, hi = fam.loci[smp]
        ro.count_stream_loci(entries.keys, entries.variant, entries.allele, vlo, vhi, b2, m1, n_pos, off, lo, hi, K,
                             counts=want[smp])
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    wres = family_results(orc, ks, want, len(fam.variants), 3, THR)
    with dkb.KmerCounter(K, n_children=3) as kc:
        kc.build_table(entries)
        kc.set_regions(vlo, vhi)
        for smp in range(ns):
            seq, qual, off = fam.reads[smp]
            _submit(dkb, kc, "submit", fam.reads[smp], smp, loci=dkb.ReadLoci(off, *fam.loci[smp]))
        got = kc.entry_counts().copy()
        res = tuple(x.copy() for x in kc.finalise(THR))
    _assert_equal(got, res, want, wres)


def test_family_finalise_from_and_overlapped_reduction(dkb):
    from denovo_kmer_b200 import dist
    fam = _family(3, seed=63)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    with dkb.KmerCounter(K, n_children=3) as kc:
        kc.build_table(entries)
        for smp in range(5):
            kc.submit(dkb.pack_reads(*fam.reads[smp], MIN_BQ), smp)
        counts = kc.entry_counts().copy()
        hits, distinct, n_kmers, calls = (x.copy() for x in kc.finalise(THR))
        ptr, n = kc.entry_counts_device()
        assert n == 5 * len(entries)
        t = dist.counts_tensor(kc)
        kc.sync()
        twice = (t * 2).contiguous()
        torch.cuda.synchronize()
        kc.finalise_launch(THR, counts_ptr=twice.data_ptr())
        hits2, distinct2, n_kmers2, calls2 = kc.results()
        assert np.array_equal(hits2, hits * 2) and np.array_equal(distinct2, distinct)
        assert np.array_equal(n_kmers2, n_kmers) and calls2.shape == calls.shape
        # one GPU, no communicator: push / flush equal plain finalise
        kc.reduce_push(THR)
        kc.reset_counts()
        kc.submit(dkb.pack_reads(*fam.reads[4], MIN_BQ), 4)
        kc.reduce_push(THR)                       # finalises the first snapshot
        red = kc.reduced_counts()
        assert red.shape == (5, len(entries)) and np.array_equal(red, counts)
        r = kc.results()
        assert all(np.array_equal(a, b) for a, b in zip(r, (hits, distinct, n_kmers, calls)))
        kc.reduce_flush(THR)
        red = kc.reduced_counts()
        assert np.array_equal(red[4], counts[4]) and red[:4].sum() == 0
    assert hits.sum() > 0


def test_family_refusals(dkb):
    from denovo_kmer_b200 import _lib
    fam = _family(2, seed=64, glen=30_000, n_var=5)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    seq, qual, off = fam.reads[0]
    st = dkb.pack_reads(seq, qual, off, MIN_BQ)
    b2 = torch.from_numpy(st.bases2.view(np.int32).copy()).cuda()
    m1 = torch.from_numpy(st.mask1.view(np.int32).copy()).cuda()
    for n_children, bad in ((1, 3), (2, 4), (6, 8)):
        with dkb.KmerCounter(K, n_children=n_children) as kc:
            kc.build_table(entries)
            for form in ("submit", "sparse", "reads", "reads4", "device"):
                for s in (bad, -1):
                    with pytest.raises(dkb.DkbError) as ei:
                        _submit(dkb, kc, form, (seq, qual, off), s)
                    assert ei.value.code == _lib.EINVAL
                    want = "sample must be 0, 1 or 2" if n_children == 1 else f"sample must be in [0, {bad})"
                    assert want in str(ei.value), str(ei.value)
            for s in (bad, -1):
                with pytest.raises(dkb.DkbError) as ei:
                    kc.submit_device_multi([(b2.data_ptr(), m1.data_ptr(), st.n_positions, 0),
                                            (b2.data_ptr(), m1.data_ptr(), st.n_positions, s)])
                assert ei.value.code == _lib.EINVAL
            kc.submit_device(b2.data_ptr(), m1.data_ptr(), st.n_positions, bad - 1)  # the last sample is fine
            assert kc.entry_counts()[bad - 1].sum() > 0 and kc.stats()["scan_launches"] == 1


RL = 150


def test_quad_full_size_analytic(dkb, orc):
    """8 Mb x 30x per sample, 2000 SNVs, a quad from the device generator with error-free
    reads, the four streams in one launch.  For every sample, an entry's count is the number
    of reads of its haplotypes that carry the entry's allele and contain its window - computed
    from the read starts with torch, not by the kernel under test or the oracle."""
    dev = torch.device("cuda:0")
    glen, n_var = 8_000_000, 2000
    genome = synth.make_genome(glen, 5)
    variants = synth.plant_variants(genome, n_var, K, 6, indel_frac=0.0, inherited_frac=0.0)
    rng = np.random.default_rng(7)
    kind = rng.integers(0, 4, size=n_var)  # 0: child 0 only, 1: child 1 only, 2: both, 3: mother + child 1
    carry = {0: (kind == 0) | (kind == 2), 3: kind != 0, 1: kind == 3, 2: np.zeros(n_var, bool)}
    for v, kd in zip(variants, kind):
        v.inherited = bool(kd == 3)
    entries = dkb.variant_kmers(synth.Trio(K, genome, variants).variant_tuples(), K)
    lut = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    ref = torch.from_numpy(lut[genome]).to(dev)
    n_reads = int(glen * 30 / RL) // 128 * 128
    pos = torch.tensor([v.pos for v in variants], device=dev)
    ev = torch.from_numpy(entries.variant.astype(np.int64)).to(dev)
    ea = torch.from_numpy(entries.allele.astype(np.int64)).to(dev)
    eu = torch.from_numpy((entries.win_index & 0x7FFF).astype(np.int64)).to(dev)
    g = pos[ev] - (K - 1) + eu
    streams, want = [], []
    for smp in range(4):
        alt = torch.from_numpy(lut[synth.apply_variants(genome, [v for v, c in zip(variants, carry[smp]) if c])]).to(dev)
        b2, m1, n_pos, _, (hap_of, starts) = synth.make_sample_device(
            [ref, alt], n_reads, RL, 90 + smp, dev, err_rate=0.0, n_rate=0.0, lowq_frac=0.0, return_meta=True)
        streams.append((b2, m1, n_pos))
        carried = torch.from_numpy(carry[smp]).to(dev)[ev]
        w = torch.zeros(len(entries), dtype=torch.int64, device=dev)
        for h in (0, 1):  # haplotype 0 = reference, 1 = this sample's alt haplotype
            s = torch.sort(starts[hap_of == h]).values
            n_in = torch.searchsorted(s, g, right=True) - torch.searchsorted(s, g + K - RL, right=False)
            allele_on_h = carried.long() if h == 1 else torch.zeros_like(ea)
            w += torch.where(ea == allele_on_h, n_in, torch.zeros_like(n_in))
        want.append(w.cpu().numpy())
    want = np.stack(want)
    torch.cuda.synchronize()
    with dkb.KmerCounter(K, n_children=2) as kc:
        kc.build_table(entries)
        kc.submit_device_multi([(b.data_ptr(), m.data_ptr(), n, smp) for smp, (b, m, n) in enumerate(streams)])
        got = kc.entry_counts().astype(np.int64)
        res = kc.finalise(THR)
    assert np.array_equal(got, want), f"{(got != want).sum()} entries differ"
    assert want.sum() > 400_000
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    wres = family_results(orc, ks, want.astype(np.uint64), n_var, 2, THR)
    _assert_equal(got, res, want.astype(np.uint64), wres)
    calls = res[3]
    # error-free reads at 30x: every child's own de novo variants are called, and only those
    for c, smp in ((0, 0), (1, 3)):
        denovo = carry[smp] & ~carry[1]
        assert ((calls[:, c] & 1) == 1)[denovo].mean() > 0.99 and not (calls[:, c] & 1)[~denovo].any()


# ---- two NCCL ranks (skipped on one GPU) ------------------------------------------------------
def _nccl_worker(rank, world, tmp):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import denovo_kmer_b200 as dkb
    from denovo_kmer_b200 import dist
    import oracle
    idf = os.path.join(tmp, "nccl_id")
    if rank == 0:
        with open(idf + ".tmp", "wb") as f:
            f.write(dkb.comm_unique_id())
        os.rename(idf + ".tmp", idf)
    while not os.path.exists(idf):
        time.sleep(0.01)
    uid = open(idf, "rb").read()
    fams = [_family(3, seed=300 + s, glen=80_000) for s in range(2)]
    entries = dkb.variant_kmers(fams[0].variant_tuples(), K)  # one table; step 1 brings new reads
    ks = oracle.KmerSet(entries.keys, entries.variant, entries.allele)
    got = []
    with dkb.KmerCounter(K, device=rank, n_children=3) as kc:
        kc.comm_init(uid, rank, world)
        kc.build_table(entries)
        for fam in fams:
            kc.reset_counts()
            for smp in range(5):
                seq, qual, off = fam.reads[smp]
                lo, hi = dist.shard_range(len(off) - 1, rank, world)
                a, b = int(off[lo]), int(off[hi])
                kc.submit(dkb.pack_reads(seq[a:b], qual[a:b], off[lo:hi + 1] - off[lo], MIN_BQ), smp)
            kc.reduce_push(THR)
        kc.reduce_flush(THR)
        got.append((kc.reduced_counts().copy(),) + tuple(x.copy() for x in kc.results()))
        kc.counts_allreduce()
        got.append((kc.entry_counts().copy(),) + tuple(x.copy() for x in kc.finalise(THR)))
        kc.comm_destroy()
    want = np.zeros((5, len(entries)), dtype=np.uint64)
    for smp in range(5):
        ks.count_reads(*fams[1].reads[smp], K, MIN_BQ, counts=want[smp])
    wres = family_results(oracle, ks, want, entries.n_variants, 3, THR)
    for g in got:
        _assert_equal(g[0], g[1:], want, wres)
    with open(os.path.join(tmp, f"ok{rank}"), "w") as f:
        f.write("ok")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_nccl_family(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_nccl_worker, args=(2, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")
