"""Kernel 3 (dkb_finalise_from: the counter memset, the per-variant reduction and the calls) at
100 000 candidates x 6 children, with locus classes and child sexes off and on, timed with
CUDA events on the library's scan stream.  Prints one JSON line.

    python scripts/calls_bench.py [--variants N] [--iters I]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import denovo_kmer_b200 as dkb  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, default=100_000)
    ap.add_argument("--children", type=int, default=6)
    ap.add_argument("--kmers", type=int, default=31, help="entries per allele (k-mers spanning an SNV)")
    ap.add_argument("--iters", type=int, default=200)
    a = ap.parse_args()
    nv, nc = a.variants, a.children
    n = nv * 2 * a.kmers
    entries = dkb.KmerEntries(np.arange(n, dtype=np.uint64) * np.uint64(7919) + np.uint64(12345),
                              np.repeat(np.arange(nv, dtype=np.uint32), 2 * a.kmers),
                              np.tile(np.repeat(np.array([0, 1], np.uint8), a.kmers), nv), None, None, nv)
    rng = np.random.default_rng(1)
    counts = torch.from_numpy(rng.integers(0, 4, size=(2 + nc, n)).astype(np.int32)).cuda()
    classes = rng.integers(0, 4, size=nv).astype(np.uint8)
    out = {"variants": nv, "children": nc, "entries": n, "gpu": torch.cuda.get_device_name(0)}
    with dkb.KmerCounter(31, n_children=nc) as kc:
        kc.build_table(entries, use_window_hints=False)
        st = torch.cuda.ExternalStream(kc.scan_stream())
        calls = {}
        for mode in ("off", "on", "off2", "on2"):
            if mode.startswith("on"):
                kc.set_locus_classes(classes)
                kc.set_child_sexes([i % 3 for i in range(nc)])
            else:
                kc.clear_locus_classes()
                kc.set_child_sexes(None)
            for _ in range(10):
                kc.finalise_launch(counts_ptr=counts.data_ptr())
            kc.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.iters):
                kc.finalise_launch(counts_ptr=counts.data_ptr())
            e1.record(st)
            e1.synchronize()
            out[f"finalise_ms_{mode}"] = round(e0.elapsed_time(e1) / a.iters, 4)
            calls[mode[:3]] = kc.results()[3]
        out["calls_differ"] = bool(not np.array_equal(calls["off"], calls["on"]))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
