"""Step rate of one scan launch per trio step (multi-batch submits) against one launch per batch.

Workloads:
  configs[0]    1 Mb, 30x, 100 candidates, k = 31: bench.py's device generator and seeds
                (bench.make_variants / synth.make_sample_device, as scripts/region_scan_bench.py)
  fetch         a per-candidate fetch trio: synth.make_trio_host (2 Mb, 30x, 100 candidates,
                seed 7), keeping only the reads whose true locus overlaps a +-500-base window
                around a candidate - what a caller that fetches reads per window submits.  The
                host generator is used because it gives every read's locus directly.
  configs[1]    64 Mb, 30x, 10 000 candidates, k = 31, the device generator: large batches
Windows are +-500 bases around each candidate.  Arms, each a pair (single, multi):
  ws_host       whole-stream, host memory: three dkb_batch_submit vs one dkb_batch_submit_multi
  rg_host       region mode, host memory: the same with loci
  rg_device     region mode, device-resident: three dkb_batch_submit_device vs one
                dkb_batch_submit_device_multi
  ws_sparse / rg_sparse    the flags as zero lists: three dkb_batch_submit_sparse vs one
                dkb_batch_submit_sparse_multi, whole stream / region mode
  ws_reads / rg_reads      decoded ASCII reads packed on the GPU: three dkb_batch_submit_reads vs
                one dkb_batch_submit_reads_multi (fetch workload only: the device generator
                makes packed streams, not reads)
  ws_reads4 / rg_reads4    the same from BAM 4-bit codes
  dense_sparse  one dkb_batch_submit_multi ("single") vs one dkb_batch_submit_sparse_multi
                ("multi"): the dense flags against the zero lists in one launch
Every arm reports the bytes per base its multi form copies over PCIe.  Counters are compared
within each pair, and across all arms of one counting mode (whole stream, region).
Host buffers are in pinned memory.  A step is one batch per sample; its time is a host clock from
the first submit to dkb_sync, so it includes copies, locus-index builds and launches.  Every
arm runs --warmup steps, then the arms alternate, --steps steps each, for --passes passes; the
result is steps per second (median over passes, with min and max), and the scan kernel's own
time per step from dkb_stats scan_ms_total.  Each arm's counters after all its steps are
compared with those of its single-submit partner, bit for bit.  Prints one JSON line with the
GPU's name and power limit read in the same run.  Needs a B200; writes nothing.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402
import denovo_kmer_b200 as dkb  # noqa: E402
from denovo_kmer_b200 import synth  # noqa: E402
from region_scan_bench import FAR, gpu_info, streams_with_loci  # noqa: E402

PAD = 500


def pinned(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).pin_memory().numpy()


def windows(n_var, variants):
    lo = np.full(n_var, FAR, dtype=np.uint64)
    hi = np.full(n_var, FAR + 1, dtype=np.uint64)
    for i, v in enumerate(variants):
        lo[i] = max(0, v.pos - PAD)
        hi[i] = v.pos + len(v.ref) + PAD
    return lo, hi


def four_bit(seq, off):
    """ASCII reads -> BAM 4-bit codes (=ACMGRSVTWYHKDBN), each read on a byte boundary."""
    lut = np.full(256, 15, dtype=np.uint8)
    for i, c in enumerate(b"=ACMGRSVTWYHKDBN"):
        lut[c] = i
        lut[ord(chr(c).lower())] = i
    codes = lut[seq]
    out = []
    for r in range(len(off) - 1):
        c = codes[int(off[r]):int(off[r + 1])]
        if len(c) % 2:
            c = np.append(c, 0)
        out.append((c[0::2] << 4) | c[1::2])
    return np.concatenate(out).astype(np.uint8) if out else np.zeros(0, np.uint8)


def extras(host, reads=None):
    """What the sparse and decoded-read arms submit, in pinned memory: the zero list of the
    stream's flags, and the decoded reads (ASCII and 4-bit) when the workload has them."""
    zoff, zbytes = dkb.mask_to_zero_list(host.mask1, host.n_positions)
    x = {"zl": (pinned(zoff), pinned(zbytes))}
    if reads is not None:
        seq, qual, off = reads
        x["reads"] = (pinned(seq), pinned(qual), pinned(off))
        x["seq4"] = pinned(four_bit(seq, off))
    return x


def device_workload(argv, dev):
    """bench.py's generator: [(device b2, device m1, host ReadStream, ReadLoci)] per sample."""
    a = bench.parse_args(argv)
    genome, variants, tuples = bench.make_variants(a, synth)
    entries = dkb.variant_kmers(tuples, a.k)
    samples = []
    for b2, m1, n_pos, n_bases, loci in streams_with_loci(a, genome, variants, dev):
        host = dkb.ReadStream(pinned(b2.cpu().numpy().view(np.uint32)), pinned(m1.cpu().numpy().view(np.uint32)),
                              int(n_pos), int(n_bases))
        samples.append((b2, m1, host, loci, extras(host)))
    return a.k, entries, windows(entries.n_variants, variants), samples


def fetch_workload(dev):
    import torch
    k = 31
    trio = synth.make_trio_host(2_000_000, 30, 100, k, seed=7)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    vlo, vhi = windows(entries.n_variants, trio.variants)
    samples = []
    for s in range(3):
        seq, qual, off = trio.reads[s]
        lo, hi = trio.loci[s]
        keep = np.zeros(len(lo), dtype=bool)
        for a, b in zip(vlo, vhi):
            keep |= (lo < b) & (hi > a)
        idx = np.nonzero(keep)[0]
        parts = [(seq[off[r]:off[r + 1]], qual[off[r]:off[r + 1]]) for r in idx]
        bseq = np.concatenate([p[0] for p in parts])
        bqual = np.concatenate([p[1] for p in parts])
        boff = np.zeros(len(idx) + 1, dtype=np.uint64)
        boff[1:] = np.cumsum([len(p[0]) for p in parts])
        st = dkb.pack_reads(bseq, bqual, boff, dkb.DEFAULT_MIN_BASEQ)
        host = dkb.ReadStream(pinned(st.bases2), pinned(st.mask1), st.n_positions, st.n_bases)
        b2 = torch.from_numpy(st.bases2.view(np.int32).copy()).to(dev)
        m1 = torch.from_numpy(st.mask1.view(np.int32).copy()).to(dev)
        samples.append((b2, m1, host, dkb.ReadLoci(boff, lo[idx], hi[idx]), extras(host, (bseq, bqual, boff))))
    torch.cuda.synchronize()
    return k, entries, (vlo, vhi), samples


ARMS = [("ws_host", False, "host"), ("rg_host", True, "host"), ("rg_device", True, "device"),
        ("ws_sparse", False, "sparse"), ("rg_sparse", True, "sparse"), ("ws_reads", False, "reads"),
        ("rg_reads", True, "reads"), ("ws_reads4", False, "reads4"), ("rg_reads4", True, "reads4"),
        ("dense_sparse", False, "dense_sparse")]
MIN_BQ = dkb.DEFAULT_MIN_BASEQ


def step_fn(kc, samples, regions, form, multi):
    loci = [x[3] for x in samples] if regions else None
    one = lambda s: loci[s] if regions else None  # noqa: E731
    smp = list(range(len(samples)))
    zl = [(x[2].bases2, *x[4]["zl"], x[2].n_positions) for x in samples]
    if form in ("reads", "reads4"):
        rd = [(x[4]["seq4"] if form == "reads4" else x[4]["reads"][0], *x[4]["reads"][1:]) for x in samples]
    if form == "dense_sparse":
        if multi:
            return lambda: kc.submit_sparse_multi(zl, smp)
        return lambda: kc.submit_multi([x[2] for x in samples], smp)
    if form == "sparse":
        if multi:
            return lambda: kc.submit_sparse_multi(zl, smp, loci=loci)
        return lambda: [kc.submit_sparse(*z[:3], z[3], s, loci=one(s)) for s, z in enumerate(zl)]
    if form in ("reads", "reads4"):
        fb = form == "reads4"
        if multi:
            return lambda: kc.submit_reads_multi(rd, smp, MIN_BQ, four_bit=fb, loci=loci)
        return lambda: [kc.submit_reads(*r, s, MIN_BQ, four_bit=fb, loci=one(s)) for s, r in enumerate(rd)]
    if multi and form == "host":
        return lambda: kc.submit_multi([x[2] for x in samples], smp, loci=loci)
    if multi:
        return lambda: kc.submit_device_multi([(x[0].data_ptr(), x[1].data_ptr(), x[2].n_positions, s)
                                               for s, x in enumerate(samples)], loci=loci)
    if form == "host":
        return lambda: [kc.submit(x[2], s, loci=one(s)) for s, x in enumerate(samples)]
    return lambda: [kc.submit_device(x[0].data_ptr(), x[1].data_ptr(), x[2].n_positions, s,
                                     loci=one(s)) for s, x in enumerate(samples)]


def pcie_bytes(samples, form):
    """Bytes the multi form of an arm copies host -> device per step (device arms: 0)."""
    n = 0
    for x in samples:
        h, e = x[2], x[4]
        if form in ("host",):
            n += h.bases2.nbytes + h.mask1.nbytes
        elif form in ("sparse", "dense_sparse"):
            n += h.bases2.nbytes + e["zl"][0].nbytes + e["zl"][1].nbytes
        elif form in ("reads", "reads4"):
            seq, qual, off = e["reads"]
            n += (e["seq4"].nbytes + 8 * (len(off) - 1) if form == "reads4" else seq.nbytes) + qual.nbytes + off.nbytes
    return n


def workload(name, k, entries, wins, samples, steps, warmup, passes):
    import torch
    counters = {}
    arms = [a for a in ARMS if a[2] not in ("reads", "reads4") or "reads" in samples[0][4]]
    for arm, regions, form in arms:
        for multi in (False, True):
            kc = dkb.KmerCounter(k)
            kc.build_table(entries)
            if regions:
                kc.set_regions(*wins)
            counters[(arm, multi)] = (kc, step_fn(kc, samples, regions, form, multi), [], [])
    for kc, fn, _, _ in counters.values():
        for _ in range(warmup):
            fn()
            kc.sync()
    for _ in range(passes):
        for kc, fn, rates, scan in counters.values():
            s0 = kc.stats()["scan_ms_total"]
            t = 0.0
            for _ in range(steps):
                t0 = time.perf_counter()
                fn()
                kc.sync()
                t += time.perf_counter() - t0
            rates.append(steps / t)
            scan.append((kc.stats()["scan_ms_total"] - s0) / steps)
    out = {"workload": name, "n_bases": int(sum(x[2].n_bases for x in samples)), "n_entries": len(entries),
           "bases_per_sample": [int(x[2].n_bases) for x in samples]}
    n_bases = sum(x[2].n_bases for x in samples)
    for arm, _, form in arms:
        res = {}
        for multi in (False, True):
            kc, _, rates, scan = counters[(arm, multi)]
            res["multi" if multi else "single"] = {
                "steps_per_s": round(float(np.median(rates)), 1), "steps_per_s_min": round(min(rates), 1),
                "steps_per_s_max": round(max(rates), 1), "scan_ms_per_step": round(float(np.median(scan)), 4)}
        a, b = counters[(arm, False)][0], counters[(arm, True)][0]
        res["counters_equal"] = bool(np.array_equal(a.entry_counts(), b.entry_counts()))
        res["counted"] = int(b.entry_counts().astype(np.uint64).sum())
        res["step_speedup"] = round(res["multi"]["steps_per_s"] / res["single"]["steps_per_s"], 3)
        res["pcie_bytes_per_base"] = round(pcie_bytes(samples, form) / n_bases, 4)
        out[arm] = res
    # every arm of one counting mode ran the same steps: its counters equal ws_host's / rg_host's
    ref = {False: counters[("ws_host", False)][0].entry_counts(), True: counters[("rg_host", False)][0].entry_counts()}
    out["counters_equal_across_arms"] = all(
        np.array_equal(counters[(arm, m)][0].entry_counts(), ref[regions]) for arm, regions, _ in arms for m in (False, True))
    for kc, _, _, _ in counters.values():
        kc.close()
    torch.cuda.synchronize()
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--no-config1", action="store_true", help="skip the large configs[1] workload")
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        sys.exit("multi_submit_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"metric": "trio_steps_per_s_multi_vs_single", **gpu_info(), "steps": args.steps, "warmup": args.warmup,
           "passes": args.passes, "results": []}
    out["results"].append(workload("configs[0]", *device_workload(["--genome-mb", "1", "--variants", "100"], dev),
                                   args.steps, args.warmup, args.passes))
    out["results"].append(workload("fetch (+-500 around 100 candidates)", *fetch_workload(dev),
                                   args.steps, args.warmup, args.passes))
    if not args.no_config1:
        out["results"].append(workload("configs[1]", *device_workload([], dev), max(2, args.steps // 10),
                                       1, args.passes))
    out["all_counters_equal"] = all(r[arm]["counters_equal"] for r in out["results"] for arm, _, _ in ARMS if arm in r)
    out["all_counters_equal_across_arms"] = all(r["counters_equal_across_arms"] for r in out["results"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
