"""Scan and finalise time of a quad (two children) in one family context, next to what it costs
as one trio context per child, in one process.

Workload: configs[1]'s shape (bench.py's genome and candidates: 64 Mb, 30x, 10 000 candidates,
k = 31), the candidates split over the two children (child c owns candidates i with i % 2 == c;
the inherited ones are carried by the mother and the owner), device-resident streams from the
bench generator: child 0, mother, father, child 1.
  family   one family context (n_children 2) with all 10 000 candidates: the four streams in
           one dkb_batch_submit_device_multi launch, then one finalise;
  trios    one trio context per child, each built on that child's own 5 000 candidates: two
           three-stream launches (the child's stream and both parents'), two finalises.
scan_ms: the library's per-launch CUDA-event time of the scan kernel (dkb_stats scan_ms_total),
per pass, over --steps passes after --warmup.  finalise_ms: CUDA events around kernel 3 on the
scan stream.  What a family saves on the host (two BAMs fewer to decode, pack and send) is not
measured here.  Prints one JSON line with the GPU's name and power limit read in the same run.
Needs a B200; writes nothing.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402
import denovo_kmer_b200 as dkb  # noqa: E402
from denovo_kmer_b200 import synth  # noqa: E402
from region_scan_bench import gpu_info  # noqa: E402

THR = dkb.DEFAULT_THRESHOLDS


def quad_streams(a, genome, variants, dev):
    """[(bases2, mask1, n_pos, n_bases)] of child 0, mother, father, child 1 (sample order)."""
    import torch
    lut = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    carried = [[v for i, v in enumerate(variants) if i % 2 == c] for c in range(2)]
    haps = {0: carried[0], 1: [v for v in variants if v.inherited], 2: [], 3: carried[1]}
    n_reads = int(len(genome) * a.depth / bench.READ_LEN) // 128 * 128
    g = torch.from_numpy(lut[genome]).to(dev)
    out = []
    for s in range(4):
        alt = torch.from_numpy(lut[synth.apply_variants(genome, haps[s])]).to(dev)
        out.append(synth.make_sample_device([g, alt], n_reads, bench.READ_LEN, 1000 + s, dev))
        del alt
    torch.cuda.synchronize()
    return out


def timed(kc, one_pass, steps, warmup):
    """(scan ms per pass, finalise ms per pass) over `steps` passes after `warmup`."""
    import torch
    stream = torch.cuda.ExternalStream(kc.scan_stream())
    fin = []
    for i in range(warmup + steps):
        if i == warmup:
            t0 = kc.stats()["scan_ms_total"]
        kc.reset_counts()
        one_pass()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        kc.finalise_launch(THR)
        e1.record(stream)
        kc.sync()
        if i >= warmup:
            fin.append(e0.elapsed_time(e1))
    return (kc.stats()["scan_ms_total"] - t0) / steps, float(np.mean(fin))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--genome-mb", type=float, default=64.0)
    ap.add_argument("--variants", type=int, default=10000)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        sys.exit("family_scan_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    a = bench.parse_args(["--genome-mb", str(args.genome_mb), "--variants", str(args.variants)])
    genome, variants, tuples = bench.make_variants(a, synth)
    streams = quad_streams(a, genome, variants, dev)
    ptrs = [(b.data_ptr(), m.data_ptr(), n, s) for s, (b, m, n, _) in enumerate(streams)]
    bases = sum(x[3] for x in streams)
    out = {"metric": "quad_scan_ms_family_vs_trios", **gpu_info(), "workload": bench.workload_name(a),
           "n_candidates": len(variants), "quad_read_bases": int(bases)}

    entries = dkb.variant_kmers(tuples, a.k)
    with dkb.KmerCounter(a.k, n_children=2) as kc:
        kc.build_table(entries)
        scan, fin = timed(kc, lambda: kc.submit_device_multi(ptrs), args.steps, args.warmup)
        family_calls = kc.results()[3].copy()
        out["family"] = {"scan_ms": round(scan, 4), "finalise_ms": round(fin, 4), "n_entries": len(entries),
                         "launches_per_pass": 1, "read_sets_scanned": 4, "tuning": list(kc.tuning())}

    out["trios"] = {"scan_ms": 0.0, "finalise_ms": 0.0, "launches_per_pass": 2, "read_sets_scanned": 6,
                    "per_child": []}
    same_calls = True
    for c in range(2):
        own = [i for i in range(len(variants)) if i % 2 == c]
        e = dkb.variant_kmers([tuples[i] for i in own], a.k)
        with dkb.KmerCounter(a.k) as kc:
            kc.build_table(e)
            trio = [ptrs[synth.child_sample(c)][:3] + (0,), ptrs[1], ptrs[2]]
            scan, fin = timed(kc, lambda: kc.submit_device_multi(trio), args.steps, args.warmup)
            same_calls &= bool(np.array_equal(kc.results()[3], family_calls[own, c]))
            out["trios"]["per_child"].append({"scan_ms": round(scan, 4), "finalise_ms": round(fin, 4),
                                              "n_entries": len(e), "tuning": list(kc.tuning())})
        out["trios"]["scan_ms"] += scan
        out["trios"]["finalise_ms"] += fin
    for key in ("scan_ms", "finalise_ms"):
        out["trios"][key] = round(out["trios"][key], 4)
    out["family_over_trios_scan"] = round(out["family"]["scan_ms"] / out["trios"]["scan_ms"], 4)
    out["family_calls_equal_trio_calls"] = same_calls
    print(json.dumps(out))


if __name__ == "__main__":
    main()
