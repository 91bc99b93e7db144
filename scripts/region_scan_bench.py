"""Scan rate of region-scoped counting next to whole-stream counting, in one process.

Workloads (bench.py's generators and seeds, rank 0): configs[1] (64 Mb, 30x, 10 000 candidates,
k = 31) and the configs[2] WGS shard (128 Mb of 30x reads, 4 000 local candidates in a 100 000-
candidate table).  Each is scanned in four modes on the same device-resident streams:
  whole      whole-stream counting
  pm500      region mode, windows of +-500 bases around each local candidate
  pm5000     region mode, +-5 000 bases
  cover      region mode, every window covering every read: the cost of the gate alone
The table's candidates of other regions get windows far from this shard's reads.  Every mode
submits one launch per sample (dkb_batch_submit_device), so the modes differ only in the gate.
The time is the library's per-launch CUDA-event time of the scan kernel (dkb_stats
scan_ms_total) over --steps passes after --warmup; building the read-locus index and copying
the loci are not in it.  Prints one JSON line, with the GPU's name and power limit read in the
same run.  Needs a B200; writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import denovo_kmer_b200 as dkb  # noqa: E402
from denovo_kmer_b200 import synth  # noqa: E402

FAR = 1 << 40  # coordinates of the table's candidates that lie in other regions


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        pass
    return info


def streams_with_loci(a, genome, variants, dev):
    """bench.make_streams' three samples (same seeds), each with its reads' loci."""
    import torch
    lut = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    mother_var = [v for v in variants if v.inherited]
    haps = [[genome, synth.apply_variants(genome, variants)], [genome, synth.apply_variants(genome, mother_var)],
            [genome, genome]]
    refpos = [[None, synth.hap_ref_positions(genome, variants)], [None, synth.hap_ref_positions(genome, mother_var)],
              [None, None]]
    n_reads = int(len(genome) * a.depth / bench.READ_LEN) // 128 * 128
    out = []
    for s in range(3):
        hs = [torch.from_numpy(lut[h]).to(dev) for h in haps[s]]
        b2, m1, n_pos, n_bases, meta = synth.make_sample_device(hs, n_reads, bench.READ_LEN, 1000 + s, dev,
                                                                return_meta=True)
        del hs
        off, lo, hi = synth.device_read_loci(meta, refpos[s], bench.READ_LEN)
        out.append((b2, m1, n_pos, n_bases, dkb.ReadLoci(off, lo, hi)))
    torch.cuda.synchronize()
    return out


def run_mode(a, entries, streams, windows, steps, warmup):
    import torch
    with dkb.KmerCounter(a.k) as kc:
        kc.build_table(entries)
        if windows is not None:
            kc.set_regions(*windows)

        def one_pass():
            kc.reset_counts()
            for s, (b2, m1, n_pos, _, loci) in enumerate(streams):
                kc.submit_device(b2.data_ptr(), m1.data_ptr(), n_pos, s, loci=None if windows is None else loci)
            kc.sync()

        for _ in range(warmup):
            one_pass()
        t0 = kc.stats()["scan_ms_total"]
        for _ in range(steps):
            one_pass()
        ms = (kc.stats()["scan_ms_total"] - t0) / steps
        counts = kc.entry_counts().copy()
        tun = kc.tuning()
    torch.cuda.synchronize()
    bases = sum(x[3] for x in streams)
    return {"scan_ms": round(ms, 4), "bases_per_s": bases / (ms * 1e-3), "tuning": list(tun)}, counts


def workload(name, a, steps, warmup, dev):
    import torch
    genome, variants, tuples = bench.make_variants(a, synth)
    entries = dkb.variant_kmers(tuples, a.k)
    streams = streams_with_loci(a, genome, variants, dev)
    n_var, n_loc = entries.n_variants, len(variants)

    def around(pad):
        lo = np.full(n_var, FAR, dtype=np.uint64)
        hi = np.full(n_var, FAR + 1, dtype=np.uint64)
        for i, v in enumerate(variants):
            lo[i] = max(0, v.pos - pad)
            hi[i] = v.pos + len(v.ref) + pad
        return lo, hi

    modes = {"whole": None, "pm500": around(500), "pm5000": around(5000),
             "cover": (np.zeros(n_var, np.uint64), np.full(n_var, 1 << 63, np.uint64))}
    res, counts = {}, {}
    for m, w in modes.items():
        res[m], counts[m] = run_mode(a, entries, streams, w, steps, warmup)
    out = {"workload": name, "n_bases": int(sum(x[3] for x in streams)), "n_entries": len(entries),
           "local_candidates": n_loc, **res,
           "cover_equals_whole": bool(np.array_equal(counts["cover"], counts["whole"])),
           "pm500_hits_fraction": float(counts["pm500"].sum() / max(counts["whole"].sum(), 1))}
    for m in ("pm500", "pm5000", "cover"):
        out[m]["rate_vs_whole"] = round(res[m]["bases_per_s"] / res["whole"]["bases_per_s"], 4)
    del streams
    torch.cuda.empty_cache()
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--no-wgs", action="store_true", help="configs[1] only")
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        sys.exit("region_scan_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"metric": "scan_bases_per_s_region_vs_whole", **gpu_info(), "results": []}
    out["results"].append(workload("configs[1]", bench.parse_args([]), args.steps, args.warmup, dev))
    if not args.no_wgs:
        a = bench.parse_args(["--genome-mb", "128", "--variants", "4000", "--table-variants", "100000"])
        out["results"].append(workload("configs[2] shard", a, args.steps, args.warmup, dev))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
