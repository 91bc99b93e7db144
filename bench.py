#!/usr/bin/env python
"""bench.py — read bases k-mer-probed per second on the BASELINE.json workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one synthetic trio shard: counts reset, the three
samples' packed read streams scanned by ONE launch of kernel 2 against the spanning-k-mer
table, (N>1: ONE NCCL sum-allreduce of the per-entry counters, made by libdkb.so on a side
stream under the next step's scan: dkb_reduce_push), kernel 3 (per-variant reduce + de novo
thresholds).  Default workload = BASELINE.json configs[1]: synthetic 30x trio, chr20-scale
(64 Mb), 10k candidate DNMs, k=31, 150 bp reads — per GPU (weak scaling: every rank holds
its own 64 Mb-scale shard of reads, the table is replicated).  `--scaling strong` splits ONE
such trio over the ranks instead.

  value         whole-job read bases / s, inputs resident in HBM (device-timed)
  e2e           same metric through the C ABI with HOST (pinned) buffers: H2D copies of
                every batch and the D2H read of the results inside the timed region
  roofline      scan kernel only: streamed bytes per launch / mean CUDA-event launch time,
                against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle port (oracle/, all host threads) on the SAME packed streams the
                GPU scanned (the full step when it fits the time bound), rank 0 at N=1 only;
                its counts are also compared with the GPU's (`matches_gpu`)
  checks        reduced == sum over ranks of the per-rank counters (N>1), taken outside the
                timed region; end-to-end run == device-resident run
  wgs_shard     the same measurement on one shard per GPU of BASELINE.json configs[2] (the
                shape north_star's targets are quoted on): 128 Mb of 30x reads per GPU against
                the replicated 100 000-candidate table, a 74 MB all-reduce per step
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "read_bases_kmer_probed_per_sec"
UNIT = "bases/s"
READ_LEN = 150
THRESHOLDS = (3, 2, 0, 1)


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genome-mb", type=float, default=64.0, help="region size per GPU, Mb")
    ap.add_argument("--depth", type=float, default=30.0)
    ap.add_argument("--variants", type=int, default=10000, help="candidates inside this GPU's region")
    ap.add_argument("--table-variants", type=int, default=0,
                    help="total candidates in the replicated table (>= --variants): the extra ones lie "
                         "in other regions of a larger genome, as for one GPU's shard of a WGS job")
    ap.add_argument("--indel-frac", type=float, default=0.0)
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank holds its own region of reads; strong: one region's reads "
                         "are split over the ranks")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="time bound of the cpu_baseline leg")
    ap.add_argument("--ref-seconds", type=float, default=150.0,
                    help="--impl reference: time bound of the whole run (the per-step sample shrinks to fit)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-wgs", action="store_true", help="skip the configs[2]-shard measurement")
    ap.add_argument("--separate-launches", action="store_true", help="one launch per sample instead of one per trio")
    ap.add_argument("--tuning", default="", help="seed_len,stride,bloom_hashes[,filter_mode] (default auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (per-entry counters, per-variant hits, "
                         "distinct, n_kmers, calls; wgs_shard_* for the configs[2] leg; --impl reference: the "
                         "counters) as DIR/<name>.npy in "
                         "float64, at most 64 MB in all: an output too large for that keeps a fixed, seeded "
                         "sample of its entries or variants, in order")
    a = ap.parse_args(argv)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def workload_name(a):
    extra = f" of {a.table_variants} in the table" if a.table_variants > a.variants else ""
    return (f"synthetic {a.depth:g}x trio, {a.genome_mb:g} Mb region per GPU, {READ_LEN} bp reads, "
            f"{a.variants} candidate DNMs{extra}, k={a.k}")


def load_synth():
    """denovo_kmer_b200/synth.py (data generation only) loaded by path, so that the reference
    arm never imports the product package."""
    spec = importlib.util.spec_from_file_location("dkb_synth", os.path.join(ROOT, "denovo_kmer_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["dkb_synth"] = mod  # dataclasses look their module up
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------
def make_variants(a, synth):
    """Genome, this region's candidates and the (left, ref, alt, right) tuples of the whole
    table — identical on every rank."""
    glen = int(a.genome_mb * 1e6)
    genome = synth.make_genome(glen, seed=1)
    variants = synth.plant_variants(genome, a.variants, a.k, seed=2, indel_frac=a.indel_frac)
    tuples = synth.Trio(a.k, genome, variants).variant_tuples()
    extra = max(0, a.table_variants - a.variants)
    if extra:  # candidates of other regions: same model, sequence this shard's reads never contain
        other = synth.make_genome(max(int(extra * 400), 1_000_000), seed=7)
        tuples += synth.Trio(a.k, other, synth.plant_variants(other, extra, a.k, seed=8,
                                                              indel_frac=a.indel_frac)).variant_tuples()
    return genome, variants, tuples


def make_streams(a, synth, genome, variants, dev, rank=0, world=1):
    """The three samples' packed streams, generated in `dev` memory: [(bases2, mask1, n_pos, n_bases)]."""
    import torch
    lut = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    g_codes = torch.from_numpy(lut[genome]).to(dev)
    child_alt = torch.from_numpy(lut[synth.apply_variants(genome, variants)]).to(dev)
    mother_alt = torch.from_numpy(
        lut[synth.apply_variants(genome, [v for v in variants if v.inherited])]).to(dev)
    n_reads = int(len(genome) * a.depth / READ_LEN) // 128 * 128
    if a.scaling == "strong":  # one region's reads split over the ranks
        n_reads = n_reads // world // 128 * 128
    haps = [[g_codes, child_alt], [g_codes, mother_alt], [g_codes, g_codes]]
    chunk = 1 << 20 if dev.type == "cuda" else 1 << 16
    return [synth.make_sample_device(haps[s], n_reads, READ_LEN, 1000 + 10 * rank + s, dev, chunk_reads=chunk)
            for s in range(3)]


def oracle_pass(ks, host_streams, k, n_entries, threads, frac=1.0):
    """One pass of the CPU oracle over (a leading fraction of) the packed streams."""
    counts = np.zeros((3, n_entries), dtype=np.uint64)
    bases = 0
    for s, (b2, m1, n_pos, n_bases) in enumerate(host_streams):
        n_reads = n_pos // (READ_LEN + 1)
        take = max(128, int(n_reads * frac) // 128 * 128) if frac < 1.0 else n_reads
        take = min(take, n_reads)
        ks.count_stream(b2, m1, take * (READ_LEN + 1), k, counts=counts[s], threads=threads)
        bases += take * READ_LEN
    return counts, bases


def run_reference(a):
    """--impl reference: the reference's CPU path on the box's host cores — the oracle port
    (jlanej/denovo_kmer's Rust source is neither mounted nor buildable here), every host
    thread, on the SAME workload (config, generator and seeds of the other arm's rank 0); each
    step is the whole trio pass unless the time bound asks for a leading fraction of the reads.
    Loads oracle/libdnk_oracle.so only — nothing of the product."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch
    import oracle
    synth = load_synth()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))) if torch.cuda.is_available() else torch.device("cpu")
    genome, variants, tuples = make_variants(a, synth)
    keys, var, al, _, _ = oracle.variant_entries(tuples, a.k)
    ks = oracle.KmerSet(keys, var, al)
    streams = make_streams(a, synth, genome, variants, dev)  # data generation only
    host = [(b2.cpu().numpy(), m1.cpu().numpy(), n_pos, nb) for (b2, m1, n_pos, nb) in streams]
    del streams
    cores = os.cpu_count() or 1
    # bound the run: calibrate on 1/16 of the step, then size the per-step sample
    t0 = time.perf_counter()
    _, nb = oracle_pass(ks, host, a.k, len(keys), cores, frac=1 / 16)
    rate = nb / (time.perf_counter() - t0)
    full_bases = sum(h[3] for h in host)
    frac = min(1.0, a.ref_seconds * rate / (full_bases * (a.steps + min(a.warmup, 1))))
    for _ in range(min(a.warmup, 1)):
        oracle_pass(ks, host, a.k, len(keys), cores, frac)
    t0 = time.perf_counter()
    bases = 0
    for _ in range(max(1, a.steps)):
        counts, nb = oracle_pass(ks, host, a.k, len(keys), cores, frac)
        bases += nb
    el = time.perf_counter() - t0
    value = bases / el
    sample = (f"{max(1, a.steps)} steps x {'the whole step' if frac >= 1.0 else f'the first {frac:.3f} of every sample of the step'} "
              f"({nb / 1e9:.2f} Gbases per step of {full_bases / 1e9:.2f}) against the full {len(keys)}-entry table; "
              f"oracle/dnk_oracle.c orc_count_stream, OpenMP, {cores} threads; {int(counts.sum())} k-mer hits per step")
    res = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": el / max(1, a.steps) * 1e3,
        "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": workload_name(a), "step_fraction": frac,
                   "reference": "CPU oracle port (oracle/dnk_oracle.c, OpenMP); jlanej/denovo_kmer's Rust source "
                                "is not mounted and no Rust toolchain exists here"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if a.dump_outputs:  # the counters of the last step's sample of the reads
        res["dumped_outputs"] = dump_outputs(a.dump_outputs, [{"counts": (counts, 1)}])
    print(json.dumps(res))


# ------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.th.join(timeout=2)
        sm, busy, mx, reasons = [], [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            try:  # "under load": the GPU was busy in that sample's window
                if float(r[7]) >= 50:
                    busy.append(sm[-1])
            except (ValueError, IndexError):
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        use = busy or sm
        return {"sm_mhz": float(np.median(use)) if use else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(busy)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_traffic(name):
    try:
        with open(os.path.join(ROOT, "profiles", "scan_traffic.json")) as f:
            return json.load(f).get(name)
    except (OSError, ValueError):
        return None


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, groups, budget=DUMP_BYTES):
    """--dump-outputs: groups = [{name: (array, axis)}] in priority order, `axis` the one that runs
    over entries or variants.  A group that fits what is left of the budget is written whole;
    otherwise every array of it keeps the same fraction of its `axis` (a sorted sample drawn with a
    fixed seed, so that two runs keep the same indices).  -> {name: [shape, stored shape]}"""
    os.makedirs(out_dir, exist_ok=True)
    left, done = budget // 8, {}  # in float64 elements; a file's .npy header takes 16 of them
    for group in groups:
        total = sum(arr.size for arr, _ in group.values())
        frac = min(1.0, max(left - 16 * len(group), 0) / max(total, 1))
        for name, (arr, axis) in group.items():
            n = arr.shape[axis]
            keep = min(n, int(n * frac))
            if keep < n:
                idx = np.sort(np.random.default_rng(12345).choice(n, keep, replace=False))
                arr = np.take(arr, idx, axis=axis)
            out = np.ascontiguousarray(arr, dtype=np.float64)
            np.save(os.path.join(out_dir, name + ".npy"), out)
            left -= out.size + 16
            done[name] = [list(np.shape(group[name][0])), list(out.shape)]
    return done


def job_outputs(prefix, counts, results):
    """What a caller of the step receives: the [3, n_entries] counters and finalise's per-variant
    hits [nv, 2, 3], distinct [nv, 2, 3], n_kmers [nv, 2] and calls [nv]."""
    hits, distinct, n_kmers, calls = results
    return {prefix + "counts": (counts, 1), prefix + "hits": (hits, 0), prefix + "distinct": (distinct, 0),
            prefix + "n_kmers": (n_kmers, 0), prefix + "calls": (calls, 0)}


class Job:
    """One workload on this rank: table, resident streams, counter, step function."""

    def __init__(self, a, rank, world, local, tdist):
        import torch
        import denovo_kmer_b200 as dkb
        from denovo_kmer_b200 import dist, synth
        self.a, self.rank, self.world, self.tdist, self.torch = a, rank, world, tdist, torch
        self.dev = torch.device("cuda", local)
        self.genome, self.variants, tuples = make_variants(a, synth)
        self.entries = dkb.variant_kmers(tuples, a.k)
        self.streams = make_streams(a, synth, self.genome, self.variants, self.dev, rank, world)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        self.bases_per_step = sum(st[3] for st in self.streams)
        self.stream_bytes = sum(st[0].numel() * 4 for st in self.streams)
        self.mask_bytes = sum(st[1].numel() * 4 for st in self.streams)
        tuning = tuple(int(x) for x in a.tuning.split(",")) if a.tuning else None
        self.kc = dkb.KmerCounter(a.k, device=local, tuning=tuning)
        self.numa_node = self.kc.bind_thread_near_gpu()
        dist.bootstrap_comm(self.kc, rank, world)  # NCCL id handed round; the communicator lives in libdkb.so
        self.kc.build_table(self.entries)
        self.ext = torch.cuda.ExternalStream(self.kc.scan_stream(), device=self.dev)

    def submit_resident(self):
        """All three samples in one launch (several when a sample exceeds one launch's 2^32 positions)."""
        kc = self.kc
        max_reads = ((1 << 32) - 4096) // (READ_LEN + 1) // 128 * 128
        per = max_reads * (READ_LEN + 1)
        if all(n_pos <= per for (_, _, n_pos, _) in self.streams) and not self.a.separate_launches:
            kc.submit_device_multi([(b2.data_ptr(), m1.data_ptr(), n_pos, s)
                                    for s, (b2, m1, n_pos, _) in enumerate(self.streams)])
            return
        for s, (b2, m1, n_pos, _) in enumerate(self.streams):
            for p0 in range(0, n_pos, per):
                kc.submit_device(b2.data_ptr() + p0 // 4, m1.data_ptr() + p0 // 8, min(per, n_pos - p0), s)

    def step(self, last=True):
        kc = self.kc
        kc.reset_counts()  # (queued behind the previous step's snapshot on the scan stream)
        self.submit_resident()
        if self.world == 1:
            kc.finalise_launch(THRESHOLDS)
        else:
            # snapshot + ncclAllReduce on the library's side stream; kernel 3 of the previous
            # step is queued behind this step's scan
            kc.reduce_push(THRESHOLDS)
            if last:
                kc.reduce_flush(THRESHOLDS)

    def barrier(self):
        if self.world > 1:
            self.tdist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, steps, warmup):
        """-> (ms max over ranks, stats before, stats after)"""
        torch = self.torch
        for _ in range(warmup):
            self.step()
        self.barrier()
        s0 = self.kc.stats()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record(self.ext)
        for i in range(steps):
            self.step(last=i == steps - 1)
        ev1.record(self.ext)
        self.barrier()
        ms = ev0.elapsed_time(ev1)
        s1 = self.kc.stats()
        t_ms = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.tdist.all_reduce(t_ms, op=self.tdist.ReduceOp.MAX)
        return float(t_ms.item()), s0, s1

    def final_counts(self):
        """Counters the last finalise saw: the sum over ranks (N>1), else this rank's own."""
        return (self.kc.reduced_counts() if self.world > 1 else self.kc.entry_counts()).copy()

    def check_sum_of_ranks(self, reduced):
        """Outside the timed region: every rank scans its shard once more WITHOUT the reduction,
        the per-rank counters are gathered (torch.distributed: the checker, not the product) and
        their sum must equal what the library's allreduce produced."""
        if self.world == 1:
            return None
        torch, tdist = self.torch, self.tdist
        self.kc.reset_counts()
        self.submit_resident()
        own = torch.from_numpy(self.kc.entry_counts().astype(np.int64)).to(self.dev)
        parts = [torch.empty_like(own) for _ in range(self.world)]
        tdist.all_gather(parts, own)
        total = torch.stack(parts).sum(0).cpu().numpy().astype(np.uint32)
        ok = torch.tensor([int(np.array_equal(total, reduced))], device=self.dev)
        tdist.all_reduce(ok, op=tdist.ReduceOp.MIN)
        return bool(ok.item())

    def roofline(self, s0, s1, steps, traffic_key):
        launches = s1["scan_launches_timed"] - s0["scan_launches_timed"]
        scan_ms = (s1["scan_ms_total"] - s0["scan_ms_total"]) / max(launches, 1)
        # what the kernel must stream: the 2-bit bases, and - when its lookups are gated by the
        # flags (dkb_stats.gated_lookups) - the 1-bit flag stream as well
        gated = bool(s1.get("gated_lookups", 0))
        per_step = self.stream_bytes + (self.mask_bytes if gated else 0)
        bytes_per_launch = per_step / max(launches / max(steps, 1), 1)
        peak, peak_src = measured_peak_gbs()
        achieved = bytes_per_launch / (scan_ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": profile_traffic(traffic_key), "kernel": "dkb::k_scan",
                "peak_source": peak_src, "launch_ms": scan_ms, "bytes_per_launch": bytes_per_launch,
                "launches_per_step": launches / max(steps, 1), "gated_lookups": gated,
                "note": ("bytes = 2-bit base stream + 1-bit flag stream (0.3775 B/read base incl. separators): the "
                         "kernel reads both in full (lookups gated by the flags)" if gated else
                         "bytes = 2-bit base stream only (0.2517 B/read base incl. separators); the 1-bit flag "
                         "stream is read only for verified seed hits") + "; all three samples of the step in one launch"}

    def close(self):
        self.kc.close()


def run_ours(a):
    import torch
    import torch.distributed as tdist
    from denovo_kmer_b200 import dist

    rank, world, local = dist.env_rank_world()
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # torch.distributed is the launcher's plumbing here: barriers, the max over ranks of the
        # timings, handing the NCCL id round, and the checks.  The counters are summed by
        # libdkb.so's own communicator.  (NCCL_DEBUG is left as the caller set it; whatever
        # NCCL prints on fd 1 goes to stderr, see main().)
        tdist.init_process_group("nccl", device_id=dev)

    job = Job(a, rank, world, local, tdist)
    kc = job.kc
    sampler = ClockSampler(local)
    if rank == 0:  # clocks are sampled from the warm-up steps on: the timed region (tens of ms)
        sampler.start()  # and, in the same record, the e2e and wgs_shard legs that follow it
        time.sleep(0.1)
    ms_max, s0, s1 = job.timed(a.steps, max(a.warmup, 3))
    n_clock_timed = len(sampler.rows)
    total_bases = job.bases_per_step * world  # weak: N shards; strong: the split trio's parts
    value = total_bases * a.steps / (ms_max * 1e-3)
    hits, distinct, n_kmers, calls = kc.results()
    ref_counts = job.final_counts()
    dump = [job_outputs("", ref_counts, (hits, distinct, n_kmers, calls))]
    sum_ok = job.check_sum_of_ranks(ref_counts)
    roof = job.roofline(s0, s1, a.steps, "dram_bytes_per_launch")
    comm = kc.comm_info() if world > 1 else None

    # ---- cpu_baseline (rank 0, N = 1): the oracle on the very streams the GPU scanned ----
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        import oracle
        e = job.entries
        ks = oracle.KmerSet(e.keys, e.variant, e.allele)
        host = [(b2.cpu().numpy(), m1.cpu().numpy(), n_pos, nb) for (b2, m1, n_pos, nb) in job.streams]
        cores = os.cpu_count() or 1
        t0 = time.perf_counter()
        _, nb = oracle_pass(ks, host, a.k, len(e), cores, frac=1 / 16)
        rate = nb / (time.perf_counter() - t0)
        frac = min(1.0, a.cpu_seconds * rate / job.bases_per_step)
        t0 = time.perf_counter()
        want, nb = oracle_pass(ks, host, a.k, len(e), cores, frac)
        el = time.perf_counter() - t0
        if frac >= 1.0:
            got = ref_counts
        else:  # the GPU on the same leading fraction (outside every timed region)
            kc.reset_counts()
            for s, (b2, m1, n_pos, _) in enumerate(job.streams):
                take = min(max(128, int(n_pos // (READ_LEN + 1) * frac) // 128 * 128), n_pos // (READ_LEN + 1))
                kc.submit_device(b2.data_ptr(), m1.data_ptr(), take * (READ_LEN + 1), s)
            got = kc.entry_counts()
        cpu = {"value": nb / el, "unit": UNIT, "cores": cores, "kind": "port",
               "matches_gpu": bool(np.array_equal(got.astype(np.uint64), want)),
               "kmer_hits": int(want.sum()),
               "sample": f"{'the whole step' if frac >= 1.0 else f'the first {frac:.3f} of every sample'}: "
                         f"{nb / 1e9:.2f} Gbases in {el:.1f} s, the packed streams the GPU scanned (D2H), against the "
                         f"full {len(e)}-entry table; oracle/dnk_oracle.c orc_count_stream with OpenMP"}
        del host, ks

    # ---- e2e: host pinned buffers through the C ABI, copies inside the timed region ----
    e2e = None
    if not a.no_e2e:
        host = []
        for (b2, m1, n_pos, _) in job.streams:  # page-locked, on the GPU's NUMA node (dkb_host_alloc)
            hb, hm = kc.host_alloc(b2.numel()), kc.host_alloc(m1.numel())
            torch.from_numpy(hb.view(np.int32)).copy_(b2)
            torch.from_numpy(hm.view(np.int32)).copy_(m1)
            host.append((hb, hm, n_pos))
        job.streams = None
        torch.cuda.empty_cache()
        reads_per_batch = 4_194_304  # 2^22 reads: batches start on 2048-position block boundaries
        pos_per_batch = reads_per_batch * (READ_LEN + 1)
        import denovo_kmer_b200 as dkb_pkg
        # the same batches with their flags as zero lists (dkb_mask_to_zero_list): what the
        # headline e2e sends; the dense-flag form is measured beside it
        sparse = []
        for s_, (hb, hm, n_pos) in enumerate(host):
            for p0 in range(0, n_pos, pos_per_batch):
                n = min(pos_per_batch, n_pos - p0)
                zoff, zbytes = dkb_pkg.mask_to_zero_list(hm[p0 // 32: p0 // 32 + (n + 127) // 128 * 4], n)
                pz = kc.host_alloc(len(zoff))
                pz[:] = zoff
                pb = kc.host_alloc((len(zbytes) + 3) // 4).view(np.uint8)[: len(zbytes)]
                pb[:] = zbytes
                sparse.append((s_, hb[p0 // 16:], pz, pb, n))
        sparse_bytes = job.stream_bytes + sum(z.nbytes + b.nbytes for (_, _, z, b, _) in sparse)

        def e2e_step(dense):
            kc.reset_counts()
            if dense:
                for s, (hb, hm, n_pos) in enumerate(host):
                    for p0 in range(0, n_pos, pos_per_batch):
                        n = min(pos_per_batch, n_pos - p0)
                        kc._ck(kc._L.dkb_batch_submit(kc._h, hb.ctypes.data + p0 // 4, hm.ctypes.data + p0 // 8, n, s))
            else:
                for (s, hb, pz, pb, n) in sparse:
                    kc._ck(kc._L.dkb_batch_submit_sparse(kc._h, hb.ctypes.data, pz.ctypes.data, pb.ctypes.data,
                                                         len(pb), n, s))
            kc.counts_allreduce()  # N>1: ncclAllReduce on the scan stream; no-op on one GPU
            return kc.finalise(THRESHOLDS)  # kernel 3 + D2H of hits/distinct/n_kmers/calls

        def e2e_timed(dense):
            e2e_step(dense)
            job.barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(job.ext)
            t0 = time.perf_counter()
            for _ in range(a.e2e_steps):
                res = e2e_step(dense)
            ev1.record(job.ext)
            own_s = time.perf_counter() - t0  # this rank's own steps (results fetched: all copies done)
            job.barrier()
            wall = time.perf_counter() - t0
            t_e = torch.tensor([max(ev0.elapsed_time(ev1) * 1e-3, wall)], dtype=torch.float64, device=dev)
            nbytes = (job.stream_bytes + job.mask_bytes) if dense else sparse_bytes
            h2d_rate = torch.tensor([nbytes * a.e2e_steps / own_s / 1e9], dtype=torch.float64, device=dev)
            rates = [h2d_rate.clone() for _ in range(world)]
            if world > 1:
                tdist.all_reduce(t_e, op=tdist.ReduceOp.MAX)
                tdist.all_gather(rates, h2d_rate)
            same = bool(np.array_equal(kc.entry_counts(), ref_counts))
            return {"value": total_bases * a.e2e_steps / float(t_e.item()), "unit": UNIT,
                    "h2d_bytes_per_step": int(nbytes), "d2h_bytes_per_step": int(sum(x.nbytes for x in res)),
                    "steps": a.e2e_steps, "counts_equal_device_resident_run": same,
                    "h2d_gbs_per_rank": [round(float(r.item()), 2) for r in rates]}

        # the box's H2D ceiling for this job: every rank copies its pinned batches to the device
        # at once, nothing else running (torch copy = cudaMemcpyAsync; not the product path)
        dst = torch.empty(max(h[0].size for h in host), dtype=torch.int32, device=dev)
        job.barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            for (hb, hm, _) in host:
                dst[: hb.size].copy_(torch.from_numpy(hb.view(np.int32)), non_blocking=True)
                dst[: hm.size].copy_(torch.from_numpy(hm.view(np.int32)), non_blocking=True)
        torch.cuda.synchronize()
        ceil_rate = torch.tensor([2 * (job.stream_bytes + job.mask_bytes) / (time.perf_counter() - t0) / 1e9],
                                 dtype=torch.float64, device=dev)
        ceils = [ceil_rate.clone() for _ in range(world)]
        if world > 1:
            tdist.all_gather(ceils, ceil_rate)
        del dst

        dense_e2e = e2e_timed(True)
        e2e = e2e_timed(False)
        e2e["flags"] = "zero list (dkb_batch_submit_sparse): %.4f bytes per read base over PCIe" % (
            sparse_bytes / job.bases_per_step)
        e2e["dense_flags"] = {k_: dense_e2e[k_] for k_ in ("value", "h2d_bytes_per_step", "h2d_gbs_per_rank",
                                                            "counts_equal_device_resident_run")}
        e2e["counts_equal_device_resident_run"] = bool(e2e["counts_equal_device_resident_run"] and
                                                        dense_e2e["counts_equal_device_resident_run"])
        e2e["h2d_ceiling_gbs_per_rank"] = [round(float(r.item()), 2) for r in ceils]
        e2e["staging"] = f"dkb_host_alloc (cudaHostAlloc on the GPU's NUMA node; rank 0: node {job.numa_node})"
        del sparse
        del host

    # ---- the feeders (f1), rank 0 at N = 1: host packer rate, and an end-to-end leg through the
    # DEVICE packer (decoded ASCII reads + quality bytes over PCIe, no per-base host work) ----
    feeders = None
    if rank == 0 and world == 1 and not a.no_e2e:
        import denovo_kmer_b200 as dkb
        from denovo_kmer_b200 import synth
        n_r = 524_288
        g = job.genome[: min(len(job.genome), 8_000_000)]
        raw = [synth.sample_reads([g, g], n_r, READ_LEN, 700 + s) for s in range(3)]
        nb = n_r * READ_LEN

        def pack_rate(threads):
            os.environ["DKB_PACK_THREADS"] = str(threads)
            seq, qual, off = raw[0]
            dkb.pack_reads(seq, qual, off, 20)
            t0 = time.perf_counter()
            for _ in range(3):
                dkb.pack_reads(seq, qual, off, 20)
            return 3 * nb / (time.perf_counter() - t0)

        def zero_list_rate(threads):  # dense flags -> zero list (what dkb_batch_submit_sparse sends)
            os.environ["DKB_PACK_THREADS"] = str(threads)
            seq, qual, off = raw[0]
            st = dkb.pack_reads(seq, qual, off, 20)
            dkb.mask_to_zero_list(st.mask1, st.n_positions)
            t0 = time.perf_counter()
            for _ in range(3):
                dkb.mask_to_zero_list(st.mask1, st.n_positions)
            return 3 * nb / (time.perf_counter() - t0)

        cores = min(os.cpu_count() or 1, 32)
        r1, rn = pack_rate(1), pack_rate(cores)
        z1, zn = zero_list_rate(1), zero_list_rate(cores)
        os.environ.pop("DKB_PACK_THREADS", None)

        pinned = []  # the BAM layer's decoded records, in page-locked buffers next to the GPU
        for (seq, qual, off) in raw:
            ps = kc.host_alloc((len(seq) + 3) // 4).view(np.uint8)[: len(seq)]
            pq = kc.host_alloc((len(qual) + 3) // 4).view(np.uint8)[: len(qual)]
            ps[:], pq[:] = seq, qual
            pinned.append((ps, pq, off))

        def reads_step():
            kc.reset_counts()
            for s, (seq, qual, off) in enumerate(pinned):
                kc.submit_reads(seq, qual, off, s, 20)
            return kc.finalise(THRESHOLDS)

        reads_step()
        t0 = time.perf_counter()
        for _ in range(5):
            reads_step()
        el = time.perf_counter() - t0
        feeders = {"host_packer_bases_per_s": {"1_thread": r1, f"{cores}_threads": rn},
                   "zero_list_bases_per_s": {"1_thread": z1, f"{cores}_threads": zn},
                   "device_packer_e2e": {"value": 5 * 3 * nb / el, "unit": UNIT,
                                         "h2d_bytes_per_base": 2.0 + 8.0 / READ_LEN,
                                         "what": "dkb_batch_submit_reads: pinned ASCII reads + quality bytes -> H2D -> "
                                                 "k_pack -> k_scan -> finalise + D2H, 3 x 524 288 reads per step"}}
        del raw

    out = None
    if rank == 0:
        st = kc.stats()
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms_max / a.steps, "higher_is_better": True,
            "scaling": a.scaling, "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {
                "workload": workload_name(a), "bases_per_step_per_gpu": int(job.bases_per_step),
                "l2": "inputs larger than L2 (%.2f GB of packed streams per step per GPU)" % (
                    (job.stream_bytes + job.mask_bytes) / 1e9),
                "table_entries": int(st["n_entries"]), "seeds": int(st["n_seeds"]),
                "tuning_seedlen_stride_hashes_filtermode": list(kc.tuning()),
                "prefilter_words": int(st.get("prefilter_words", 0)), "gated_lookups": bool(st.get("gated_lookups", 0)),
                "denovo_calls": int((calls & 1).sum()), "variants": int(len(calls)),
                "collective": ("1 ncclAllReduce(sum) of %d uint32 per step inside libdkb.so (dkb_reduce_push); "
                               "communicator of %d ranks, NCCL %d" % (3 * len(job.entries), comm[1], comm[2]))
                if world > 1 else "none",
            },
            "roofline": roof,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "feeders": feeders,
            "checks": {"reduced_equals_sum_of_ranks": sum_ok,
                       "cpu_oracle_matches_gpu": cpu["matches_gpu"] if cpu else None,
                       "e2e_equals_device_resident": e2e["counts_equal_device_resident_run"] if e2e else None},
            # per step: 1 scan launch (the trio) + k_variant_reduce + k_calls
            "gpu_launches": int((s1["scan_launches"] - s0["scan_launches"]) + 2 * a.steps),
            "clocks": None,  # filled in when the sampler stops, after the last leg
        }
    job.close()
    del job
    torch.cuda.empty_cache()

    # ---- the configs[2] shape: one WGS shard per GPU against the 100 000-candidate table ----
    if not a.no_wgs and a.table_variants == 0 and a.scaling == "weak":
        w = parse_args([])
        w.gpus, w.steps, w.warmup, w.k, w.depth = a.gpus, a.steps, a.warmup, a.k, a.depth
        w.genome_mb, w.variants, w.table_variants = 128.0, 4000, 100000
        w.separate_launches = a.separate_launches
        wj = Job(w, rank, world, local, tdist)
        ms_w, w0, w1 = wj.timed(w.steps, max(w.warmup, 3))
        red = wj.final_counts()
        if a.dump_outputs and rank == 0:
            dump.append(job_outputs("wgs_shard_", red, wj.kc.results()))
        sum_w = wj.check_sum_of_ranks(red)
        if rank == 0:
            roof_w = wj.roofline(w0, w1, w.steps, "wgs_dram_bytes_per_launch")
            stw = wj.kc.stats()
            out["wgs_shard"] = {
                "workload": workload_name(w) + " (one shard per GPU of BASELINE.json configs[2])",
                "value": wj.bases_per_step * world * w.steps / (ms_w * 1e-3), "unit": UNIT, "n_gpus": world,
                "ms_per_step": ms_w / w.steps, "scaling": "weak",
                "table_entries": int(stw["n_entries"]), "seeds": int(stw["n_seeds"]),
                "tuning_seedlen_stride_hashes_filtermode": list(wj.kc.tuning()),
                "allreduce_bytes_per_step": int(12 * len(wj.entries)) if world > 1 else 0,
                "kmer_hits_per_step": int(red.astype(np.uint64).sum()),
                "reduced_equals_sum_of_ranks": sum_w,
                "roofline": {k: roof_w[k] for k in ("achieved", "peak", "frac", "launch_ms", "bytes_per_launch", "traffic")},
            }
        wj.close()

    if rank == 0:
        out["clocks"] = sampler.stop()
        out["clocks"]["samples_by_end_of_timed_region"] = n_clock_timed
        if a.dump_outputs:
            out["dumped_outputs"] = dump_outputs(a.dump_outputs, dump)
        print(json.dumps(out))
    if world > 1:
        tdist.destroy_process_group()


def main():
    a = parse_args()
    # stdout carries the ONE JSON line and nothing else: libraries that chat on fd 1 (NCCL with
    # NCCL_DEBUG=INFO/VERSION, torch's "NCCL version ..." on the first collective) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    global print

    def print(*args, **kw):  # noqa: A001 - the module's result lines
        if kw.get("file") is not None:
            import builtins
            return builtins.print(*args, **kw)
        os.write(json_fd, (" ".join(str(x) for x in args) + "\n").encode())

    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
