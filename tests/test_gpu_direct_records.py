"""-m gpu: direct seed records (DESIGN.md §4: stage C counts a direct record's windows straight
from the record, without the key table) next to records that take the key-table path, in the
same launch: isolated SNVs (direct) beside indels, SNV pairs closer than k, keys shared by two
variants and palindromic keys, with and without window hints, in region mode with windows that
cut reads out, and in a quad family.  Counters are the oracle's bit for bit, and the number of
direct halves equals a pure-Python model of the build's rule, so a silent fall-back of every
record to the key table (or a record made direct that should not be) fails here."""
import numpy as np
import pytest

import region_oracle as ro
from denovo_kmer_b200 import synth
from family_oracle import family_counts
from helpers import gpu_counts, oracle_counts

pytestmark = pytest.mark.gpu

NB_BASES = 48
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}


def _other(base, r):
    return "ACGT"[("ACGT".index(base) + 1 + r) % 4]


def _mixed_variants(genome, k, n_var, seed):
    """Isolated SNVs and indels on a grid (plant_variants), then: an SNV 7 bases after every
    fifth SNV, carried with it (pairs closer than k); a second candidate at the locus of every
    fifth SNV with another ALT base (keys shared by two variants; not carried); for even k a
    k-base reverse-complement palindrome written over the reference around every fourth SNV
    (a palindromic key).  Returns (genome, carried variants, candidates)."""
    rng = np.random.default_rng(seed)
    genome = genome.copy()
    variants = synth.plant_variants(genome, n_var, k, seed, indel_frac=0.3)
    snvs = [v for v in variants if len(v.ref) == 1 and len(v.alt) == 1]
    if k % 2 == 0:
        for v in snvs[::4]:
            half = synth.make_genome(k // 2, int(rng.integers(1 << 30))).tobytes().decode()
            pal = half + "".join(COMP[c] for c in reversed(half))
            a = v.pos - int(rng.integers(0, k))
            genome[a:a + k] = np.frombuffer(pal.encode(), dtype=np.uint8)
        for v in variants:  # the palindromes may have rewritten a REF
            v.ref = genome[v.pos:v.pos + len(v.ref)].tobytes().decode()
            if len(v.alt) == 1 and len(v.ref) == 1 and v.alt == v.ref:
                v.alt = _other(v.ref, 0)
            elif len(v.ref) == 1 and len(v.alt) > 1:
                v.alt = v.ref + v.alt[1:]
            elif len(v.ref) > 1:
                v.alt = v.ref[0]
    pairs = [synth.Variant(v.pos + 7, chr(genome[v.pos + 7]), _other(chr(genome[v.pos + 7]), int(rng.integers(3))))
             for v in snvs[1::5]]
    shared = [synth.Variant(v.pos, v.ref, _other(v.alt, 0) if _other(v.alt, 0) != v.ref else _other(v.alt, 1))
              for v in snvs[2::5]]
    carried = sorted(variants + pairs, key=lambda v: v.pos)
    return genome, carried, sorted(carried + shared, key=lambda v: v.pos)


def _trio(k, seed, glen=120_000, depth=12, n_var=40):
    genome, carried, cands = _mixed_variants(synth.make_genome(glen, seed), k, n_var, seed + 1)
    child = synth.apply_variants(genome, carried)
    trio = synth.Trio(k, genome, cands)
    refpos = {0: [None, synth.hap_ref_positions(genome, carried)], 1: [None, None], 2: [None, None]}
    n_reads = int(len(genome) * depth / 150)
    for smp, haps in enumerate([[genome, child], [genome, genome], [genome, genome]]):
        seq, qual, off, (hap_of, starts) = synth.sample_reads(haps, n_reads, 150, seed + 10 + smp, return_meta=True)
        trio.reads[smp] = (seq, qual, off)
        trio.loci[smp] = synth.read_loci(refpos[smp], hap_of, starts, np.diff(off).astype(np.int64))
    return trio


# ---- pure-Python model of the build's rule (csrc/dkb_build.cuh, k_assign_seeds + k_finish_direct)
def _stream(key, k):
    return sum(((key >> (2 * (k - 1 - t))) & 3) << (2 * t) for t in range(k))


def _rc_stream(x, s):
    return sum((3 - ((x >> (2 * t)) & 3)) << (2 * (s - 1 - t)) for t in range(s))


def model_halves(entries, k, s, D, canon):
    """(occupied halves, direct halves) of a table built with window hints."""
    keys = [int(x) for x in entries.keys]
    var, al = entries.variant.astype(int), entries.allele.astype(int)
    wi, wc = entries.win_index.astype(int), entries.win_count.astype(int)
    seen, live = set(), []
    for i, key in enumerate(keys):  # first (key, variant, allele) wins
        live.append((key, var[i], al[i]) not in seen)
        seen.add((key, var[i], al[i]))
    owners = {}
    for i, key in enumerate(keys):
        if live[i]:
            owners[key] = owners.get(key, 0) + 1
    E, km, smask = k - s, (1 << 2 * k) - 1, (1 << 2 * s) - 1
    G = ((E + 1) // D) * D
    halves = {}
    for i, key in enumerate(keys):
        if not live[i]:
            continue
        v0 = _stream(key, k)
        v1 = ~key & km
        for ori, v in ((0, v0), (1, v1)):
            if ori == 1 and v1 == v0:
                continue
            u = wi[i] & 0x7FFF
            if ori != (wi[i] >> 15) & 1:
                u = wc[i] - 1 - u
            for c in range(D):
                r = (u + c) % D
                base = E - ((E - r) % D)
                P = base if u <= base else base + ((u - base + G - 1) // G) * G
                j = P - u
                x = (v >> (2 * j)) & smask
                flip = 0
                if canon:
                    rc = _rc_stream(x, s)
                    flip = int(rc < x)
                    x = min(x, rc)
                halves.setdefault((x, flip), []).append((i, var[i], al[i], j, v, owners[key] > 1))
    n_direct = 0
    for des in halves.values():
        if E + k > NB_BASES or any(d[5] for d in des) or len({d[1] for d in des}) > 1:
            continue
        base_at = {}  # neighbourhood position -> bases the windows show there
        for _, _, _, j, v, _ in des:
            for t in range(k):
                base_at.setdefault(E - j + t, set()).add((v >> (2 * t)) & 3)
        disputed = [q for q, b in base_at.items() if len(b) > 1]
        A = [{d[3] for d in des if d[2] == a} for a in (0, 1)]
        ok = all(not A[a] or len({d[0] - d[3] for d in des if d[2] == a}) == 1
                 or len({d[0] + d[3] for d in des if d[2] == a}) == 1 for a in (0, 1))
        if A[0] and A[1]:
            ok = ok and A[0] == A[1] and len(disputed) == 1
            if ok:
                X = disputed[0]
                shown = [{(d[4] >> (2 * (X - E + d[3]))) & 3 for d in des if d[2] == a} for a in (0, 1)]
                ok = all(E - d[3] <= X < E - d[3] + k for d in des) and all(len(b) == 1 for b in shown) \
                    and shown[0] != shown[1]
        else:
            ok = ok and not disputed
        n_direct += ok
    return len(halves), n_direct


def _check(got, want, tun):
    bad = np.nonzero(got.astype(np.uint64) != want)
    assert len(bad[0]) == 0, (tun, len(bad[0]), [(int(s), int(e), int(got[s, e]), int(want[s, e]))
                                                 for s, e in zip(*bad)][:5])
    assert want.sum() > 0


@pytest.mark.parametrize("k", [31, 30, 21])
@pytest.mark.parametrize("tuning", [None, (15, 16, 2, 2), (13, 8, 1, 2), (14, 4, 2, 2), (12, 2, 1, 1), (15, 1, 2),
                                    (15, 16, 2, 1)])
@pytest.mark.parametrize("hints", [True, False])
def test_direct_and_probed_records(dkb, orc, k, tuning, hints):
    if tuning is not None and tuning[0] > k - tuning[1] + 1:
        pytest.skip("seed does not fit this stride at this k")
    trio = _trio(k, seed=300 + k)
    entries = dkb.variant_kmers(trio.variant_tuples(), k, drop_shared=False)
    _, want = oracle_counts(orc, entries, trio, k, 20)
    got, st, tun = gpu_counts(dkb, entries, trio, k, 20, tuning=tuning, hints=hints)
    _check(got, want, tun)
    if 2 * k - tun[0] <= NB_BASES:  # the records have a neighbourhood: direct ones exist
        assert 0 < st["direct_halves"] < st["occupied_halves"], st
    else:
        assert st["direct_halves"] == 0, st
    if hints:
        occ, direct = model_halves(entries, k, tun[0], tun[1], tun[3] == 2)  # L2 filter: canonical seeds
        assert (st["occupied_halves"], st["direct_halves"]) == (occ, direct), (tun, occ, direct, st)
    if tun[1] == 16 and hints:
        # isolated SNV windows are the bulk of the table: most of its halves are direct
        assert st["direct_halves"] > 0.5 * st["occupied_halves"], st


@pytest.mark.parametrize("tuning", [None, (15, 16, 2, 2), (14, 4, 1, 2), (15, 1, 1)])
def test_direct_records_region_mode(dkb, orc, tuning):
    """Region mode with windows that cut half the reads out: the direct path counts only reads
    whose alignment overlaps the entry's variant window, as the key-table path does."""
    k, min_bq = 31, 20
    trio = _trio(k, seed=41)
    rng = np.random.default_rng(0)
    for smp in range(3):
        lo, hi = trio.loci[smp]
        far = rng.random(len(lo)) < 0.5
        lo[far] += np.uint64(1 << 30)
        hi[far] += np.uint64(1 << 30)
    entries = dkb.variant_kmers(trio.variant_tuples(), k, drop_shared=False)
    vlo, vhi = ro.windows(trio.variants, 40)
    want = np.zeros((3, len(entries)), dtype=np.uint64)
    with dkb.KmerCounter(k, tuning=tuning) as kc:
        kc.build_table(entries)
        kc.set_regions(vlo, vhi)
        for smp in range(3):
            seq, qual, off = trio.reads[smp]
            lo, hi = trio.loci[smp]
            b2, m1, n_pos = orc.pack_stream(seq, qual, off, min_bq)
            ro.count_stream_loci(entries.keys, entries.variant, entries.allele, vlo, vhi, b2, m1, n_pos, off, lo, hi,
                                 k, counts=want[smp])
            kc.submit(dkb.pack_reads(seq, qual, off, min_bq), smp, loci=dkb.ReadLoci(off, lo, hi))
        got = kc.entry_counts().copy()
        st, tun = kc.stats(), kc.tuning()
    _check(got, want, tun)
    assert 0 < st["direct_halves"] < st["occupied_halves"], st


def test_direct_records_quad_family(dkb, orc):
    """A quad (two children) against one table: every sample's counters."""
    k, min_bq = 31, 20
    fam = synth.make_family_host(120_000, 10, 40, k, 2, seed=77, indel_frac=0.3, shared_frac=0.3)
    entries = dkb.variant_kmers(fam.variant_tuples(), k)
    _, want = family_counts(orc, entries, fam, k, min_bq, 4)
    with dkb.KmerCounter(k, n_children=2) as kc:
        kc.build_table(entries)
        for smp in range(4):
            seq, qual, off = fam.reads[smp]
            kc.submit(dkb.pack_reads(seq, qual, off, min_bq), smp)
        got = kc.entry_counts().copy()
        st, tun = kc.stats(), kc.tuning()
    _check(got, want, tun)
    assert 0 < st["direct_halves"] < st["occupied_halves"], st
