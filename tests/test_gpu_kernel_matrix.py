"""-m gpu: every built instantiation of the scan kernel k_scan<D, NH, FM, PROF, RG> (132: 44
(stride, hashes, filter mode) combinations, each plain, with the profiling counters, and as a
region twin) forced one by one and compared bit for bit with the oracle on the adversarial inputs
of tests/adversarial.py; the combinations that are not built are refused.

Each kernel runs at (k 31, s 15) with window hints and at (k 30, s 14) without; each (stride,
filter mode, region) also at (k 31, s 12), where 2k - s > 48 and every seed takes stage C's
no-neighbourhood fallback.  Whole-stream kernels scan the four batches (sample 0 split in two) in
one dkb_batch_submit_device_multi launch; region twins scan one batch at a time with its loci.
The oracle runs once per input: KmerSet.count_reads, and region_oracle.count_stream_loci for
region mode.  The profiling kernels' counters are checked against what the counts imply."""
import itertools

import numpy as np
import pytest
import torch

import adversarial as adv
import region_oracle as ro

pytestmark = pytest.mark.gpu

STRIDES, HASHES = (1, 2, 4, 8, 16), (1, 2, 3, 4)
MODES = {"smem": (1, None), "l2": (2, "0"), "l2_pre": (2, "37120")}  # filter_mode, DKB_PREFILTER_WORDS
RUNS = [(31, 15, True), (30, 14, False)]
FALLBACK = (31, 12, True)  # 2k - s = 50 > 48


@pytest.fixture(scope="module")
def inputs(dkb, orc):
    out = {}
    for k in (31, 30):
        inp = adv.build(dkb, k, seed=k)
        entries = dkb.variant_kmers(inp.variants, k)
        ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
        whole = np.zeros((3, len(entries)), dtype=np.uint64)
        region = np.zeros((3, len(entries)), dtype=np.uint64)
        # valid read windows whose key is live: a KmerSet with one entry per distinct live key
        live_keys = np.unique(entries.keys[ks.live().astype(bool)])
        one = orc.KmerSet(live_keys, np.arange(len(live_keys), dtype=np.uint32), np.zeros(len(live_keys), np.uint8))
        n_live_windows = 0
        streams, dev = [], []
        for b in inp.batches:
            ks.count_reads(b.seq, b.qual, b.off, k, adv.MIN_BQ, counts=whole[b.sample])
            n_live_windows += int(one.count_reads(b.seq, b.qual, b.off, k, adv.MIN_BQ).sum())
            st = dkb.pack_reads(b.seq, b.qual, b.off, adv.MIN_BQ)
            b2, m1, n_pos = orc.pack_stream(b.seq, b.qual, b.off, adv.MIN_BQ)
            assert n_pos == st.n_positions and np.array_equal(st.bases2[:len(b2)], b2)
            ro.count_stream_loci(entries.keys, entries.variant, entries.allele, inp.vlo, inp.vhi, b2, m1, n_pos,
                                 b.off, b.lo, b.hi, k, counts=region[b.sample])
            streams.append(st)
            dev.append((torch.from_numpy(st.bases2.view(np.int32).copy()).cuda(),
                        torch.from_numpy(st.mask1.view(np.int32).copy()).cuda()))
        torch.cuda.synchronize()
        assert whole.sum() > region.sum() > 0
        out[k] = dict(inp=inp, entries=entries, whole=whole, region=region, n_live_windows=n_live_windows,
                      streams=streams, dev=dev)
    return out


def _kernel(D, NH, mode, gate, prof, rg):
    """The instantiation a combination selects, or the error code that refuses it."""
    from denovo_kmer_b200 import _lib
    if mode != "smem" and (D == 1 or NH > 2):
        return _lib.EINVAL
    if prof and rg:
        return _lib.ESTATE
    fm = 0 if mode == "smem" else (2 if mode == "l2_pre" else 1) + (2 if gate and D >= 8 else 0)
    return (D, NH, fm, prof, rg)


def _run(dkb, data, kernel, s, hints):
    D, NH, fm, prof, rg = kernel
    k = data["inp"].k
    with dkb.KmerCounter(k, tuning=(s, D, NH, 1 if fm == 0 else 2)) as kc:
        kc.build_table(data["entries"], use_window_hints=hints)
        st = kc.stats()
        assert kc.tuning() == (s, D, NH, 1 if fm == 0 else 2)
        assert (st["prefilter_words"] > 0) == (fm in (2, 4)) and st["gated_lookups"] == (fm >= 3)
        assert st["table_slots"] == adv.table_slots(len(data["entries"]))
        if prof:
            kc.profile_counters(True)
        if rg:
            inp = data["inp"]
            kc.set_regions(inp.vlo, inp.vhi)
            for b, stream in zip(inp.batches, data["streams"]):
                kc.submit(stream, b.sample, loci=dkb.ReadLoci(b.off, b.lo, b.hi))
        else:
            kc.submit_device_multi([(b2.data_ptr(), m1.data_ptr(), stream.n_positions, b.sample)
                                    for (b2, m1), stream, b in zip(data["dev"], data["streams"], data["inp"].batches)])
        got = kc.entry_counts().copy()
        kc.sync()
        st = kc.stats()
        if prof:
            kc.profile_counters(False)
            kc.profile_counters(True)
            kc.sync()
            again = kc.stats()
            st["restarted"] = all(again[f] == 0 for f in ("bloom_hits", "seed_hits", "windows_probed", "window_hits"))
    return got, st


def test_every_scan_kernel_against_the_oracle(dkb, inputs, monkeypatch):
    from denovo_kmer_b200 import _lib
    checked, failures, fallback_done = set(), [], set()
    for D, NH, mode, gate, prof, rg in itertools.product(STRIDES, HASHES, MODES, (False, True), (False, True),
                                                         (False, True)):
        kernel = _kernel(D, NH, mode, gate, prof, rg)
        fmode, pre = MODES[mode]
        if pre is None:
            monkeypatch.delenv("DKB_PREFILTER_WORDS", raising=False)
        else:
            monkeypatch.setenv("DKB_PREFILTER_WORDS", pre)
        monkeypatch.setenv("DKB_GATE", "1" if gate else "0")
        data = inputs[31]
        if isinstance(kernel, int):  # not built: refused
            with pytest.raises(_lib.DkbError) as ei:
                if kernel == _lib.ESTATE:  # the region twin's tuning, with the profiling counters on
                    _run(dkb, data, _kernel(D, NH, mode, gate, False, rg)[:3] + (prof, rg), 15, True)
                else:
                    with dkb.KmerCounter(31, tuning=(15, D, NH, fmode)) as kc:
                        kc.build_table(data["entries"])
            assert ei.value.code == kernel, (D, NH, mode, gate, prof, rg, str(ei.value))
            continue
        if kernel in checked:  # gate at D < 8 or with the shared-memory filter: ignored, same kernel
            assert gate and (D < 8 or mode == "smem")
            with dkb.KmerCounter(31, tuning=(15, D, NH, fmode)) as kc:
                kc.build_table(data["entries"])
                assert kc.stats()["gated_lookups"] == 0
            continue
        runs = list(RUNS)
        if (D, kernel[2], rg) not in fallback_done and not prof:
            runs.append(FALLBACK)
            fallback_done.add((D, kernel[2], rg))
        for k, s, hints in runs:
            s = min(s, k - D + 1)
            d = inputs[k]
            got, st = _run(dkb, d, kernel, s, hints)
            want = d["region"] if rg else d["whole"]
            bad = np.argwhere(got.astype(np.uint64) != want)
            if len(bad):
                smp, e = bad[0]
                failures.append(f"kernel {kernel} (k={k}, s={s}, hints={hints}): {len(bad)} counters differ, first "
                                f"sample {smp} entry {e}: {int(got[smp, e])} vs {int(want[smp, e])}")
            if prof:
                total = int(got.astype(np.uint64).sum())
                if not (st["window_hits"] == total and st["windows_probed"] >= d["n_live_windows"]
                        and st["seed_hits"] <= st["bloom_hits"] and st["restarted"]):
                    failures.append(f"kernel {kernel} (k={k}, s={s}): profiling counters {st} against "
                                    f"{total} counts and {d['n_live_windows']} live windows")
        checked.add(kernel)
    assert not failures, "\n".join(failures[:10])
    assert len(checked) == 132, len(checked)
    assert len(fallback_done) == 34

