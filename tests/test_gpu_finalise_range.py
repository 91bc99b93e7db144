"""-m gpu: kernel 3 (k_variant_reduce, k_calls) at the edge of its integer range.  Crafted u32
counters whose per-(variant, allele, sample) sums pass 2^32 - 1 - inside one warp's reduction,
across warps and blocks, over non-contiguous entries, at exactly 2^32 - 1 and 2^32 - go through
dkb_finalise_from and through the snapshot buffer of dkb_reduce_push / _flush, in trio and family
contexts.  The reference is the oracle's u64 sums: the GPU's hits must equal them clamped at
UINT32_MAX, distinct and n_kmers exactly, and the calls must equal the oracle's calls on the
UNclamped sums (include/dkb.h: exact for every max_parent_alt_hits below UINT32_MAX)."""
import numpy as np
import pytest
import torch

from denovo_kmer_b200 import dist
from denovo_kmer_b200.synth import child_sample
from family_oracle import family_results

pytestmark = pytest.mark.gpu

K = 31
MAX = 0xFFFFFFFF
N = 1536  # six blocks of kernel 3's 256 threads
# (min_child_alt_hits, min_child_alt_distinct, max_parent_alt_hits, min_parent_ref_hits)
THRESHOLDS = [(3, 2, 10, 1), (MAX, 2, MAX - 1, MAX)]


def _layout(n_children, seed=0):
    """(keys, variant, allele, counts uint64 [NS, N], n_variants, special variant ids)."""
    ns = 2 + n_children
    children = [0] + list(range(3, ns))
    rng = np.random.default_rng(seed)
    fwd = rng.integers(0, 1 << (2 * K), size=N, dtype=np.uint64)
    rc = np.zeros_like(fwd)
    for b in range(K):  # reverse complement of every key, two bits at a time
        rc |= (np.uint64(3) - ((fwd >> np.uint64(2 * b)) & np.uint64(3))) << np.uint64(2 * (K - 1 - b))
    keys = np.minimum(fwd, rc)
    variant = (np.arange(N) // 24).astype(np.uint32)  # filler: 64 variants, alleles of 12 entries
    allele = ((np.arange(N) // 12) % 2).astype(np.uint8)
    counts = rng.integers(0, 6, size=(ns, N)).astype(np.uint64)
    counts[:, rng.random(N) < 0.3] = 0
    nv = 64

    def group(idx, a, per_sample):
        """A new variant whose allele `a` owns entries idx; per_sample(smp, j) = count of entry j."""
        nonlocal nv
        idx = np.asarray(idx)
        variant[idx], allele[idx] = nv, a
        for smp in range(ns):
            counts[smp, idx] = [per_sample(smp, j) for j in range(len(idx))]
        nv += 1
        return nv - 1

    special = {}
    # one aligned warp: the sum of 32 counters wraps inside the warp reduction (sample 0: 2^32 exactly)
    special["warp"] = group(range(32, 64), 1, lambda smp, j: 0x08000000 + smp)
    variant[64:96], allele[64:96] = special["warp"], 0
    # warp 7 / warp 8 and block 0 / block 1: each warp's partial sum fits, their total does not
    special["straddle"] = group(range(252, 260), 1, lambda smp, j: 0x38000000 + smp)
    # one allele over every 37th entry of 20 warps, interleaved with other variants
    special["scatter"] = group(range(300, 300 + 37 * 20, 37), 0, lambda smp, j: 0x10000000 + j)
    variant[range(301, 301 + 37 * 6, 37)], allele[range(301, 301 + 37 * 6, 37)] = special["scatter"], 1
    # exactly 2^32 - 1 and exactly 2^32, each within a warp (allele 1) and across warps (allele 0)
    special["max"] = group([1100, 1101], 1, lambda smp, j: (0x80000000, 0x7FFFFFFF)[j])
    variant[[1150, 1190]], allele[[1150, 1190]] = special["max"], 0
    counts[:, 1150], counts[:, 1190] = 0x80000000, 0x7FFFFFFF
    special["2^32"] = group([1200, 1201], 1, lambda smp, j: 0x80000000)
    variant[[1230, 1290]], allele[[1230, 1290]] = special["2^32"], 0
    counts[:, 1230], counts[:, 1290] = 0x80000000, 0x80000000

    # one variant per call clause, decided on a sum that passes 2^32 - 1: a de novo candidate with
    # good child support and covered parents, except for the one saturated total
    def clause(base, samples, a, pair):
        ids = np.arange(base, base + 8)
        v = group(ids[:4], 1, lambda smp, j: 50 if smp in children else 0)  # alt
        variant[ids[4:]], allele[ids[4:]] = v, 0                              # ref
        counts[:, ids[4:]] = 20
        counts[np.ix_(samples, ids[:4] if a == 1 else ids[4:])] = pair + (0, 0)
        return v

    # exact: FATHER_ALT / MOTHER_ALT; wrapped to 3 alt hits, under max_parent_alt_hits 10: de novo
    special["father_alt"] = clause(1320, [2], 1, (0x80000002, 0x80000001))
    special["mother_alt"] = clause(1330, [1], 1, (0x80000002, 0x80000001))
    # 2^32 ref hits: exact de novo; wrapped to 0, PARENT_UNCOVERED
    special["mother_ref"] = clause(1340, [1], 0, (0x80000000, 0x80000000))
    # 2^32 alt hits in 2 distinct k-mers: exact de novo; wrapped to 0, CHILD_LOW
    special["child_alt"] = clause(1350, children, 1, (0x80000000, 0x80000000))
    # a repeated (key, variant, allele) triple is dead: its counter must not reach the sums
    keys[1400], variant[1400], allele[1400] = keys[1320], variant[1320], allele[1320]
    counts[:, 1400] = MAX
    assert counts.max() <= MAX
    return keys, variant, allele, counts, nv, special


def _oracle(orc, keys, variant, allele, counts, nv, n_children, thr):
    ks = orc.KmerSet(keys, variant, allele)
    assert ks.live()[1400] == 0
    return family_results(orc, ks, counts, nv, n_children, thr)


def _check(res, want, special, thr, wrapped_calls):
    hits, dist_, nk, calls = res
    o_hits, o_dist, o_nk, o_calls = want
    calls = calls.reshape(o_calls.shape)
    bad = np.argwhere(hits.astype(np.uint64) != np.minimum(o_hits, MAX))
    assert len(bad) == 0, f"first differing (variant, allele, sample): {tuple(bad[0])}: " \
        f"{int(hits[tuple(bad[0])])} vs {int(o_hits[tuple(bad[0])])}"
    assert np.array_equal(dist_.astype(np.uint64), o_dist) and np.array_equal(nk, o_nk)
    bad = np.argwhere(calls != o_calls)
    assert len(bad) == 0, f"first differing (variant, child): {tuple(bad[0])}, thresholds {thr}"
    # the input has teeth: sums past 2^32 - 1 in every special group, and calls that wrapping changes
    for name, v in special.items():
        if name != "max":
            assert (o_hits[v] > MAX).any(), name
    assert (o_hits[special["max"]] == MAX).all() and (o_hits[special["2^32"], :, 0] == 1 << 32).all()
    assert not np.array_equal(wrapped_calls, o_calls)


def _wrapped_calls(orc, want, n_children, thr):
    """The calls the rule gives on sums taken mod 2^32 (what a wrapping kernel 3 computes)."""
    o_hits, o_dist = want[0] % (1 << 32), want[1]
    return np.stack([orc.calls(o_hits[:, :, [child_sample(c), 1, 2]], o_dist[:, :, [child_sample(c), 1, 2]], thr)
                     for c in range(n_children)], axis=1)


@pytest.mark.parametrize("n_children", [1, 2, 6])
def test_finalise_saturates(dkb, orc, n_children):
    keys, variant, allele, counts, nv, special = _layout(n_children, seed=n_children)
    entries = dkb.KmerEntries(keys, variant, allele, n_variants=nv)
    u32 = torch.from_numpy(counts.astype(np.uint32).view(np.int32).reshape(-1)).cuda()
    with dkb.KmerCounter(K, n_children=n_children) as kc:
        kc.build_table(entries, use_window_hints=False)
        assert kc.stats()["n_live_entries"] == N - 1
        for thr in THRESHOLDS:
            want = _oracle(orc, keys, variant, allele, counts, nv, n_children, thr)
            wrapped = _wrapped_calls(orc, want, n_children, thr)
            torch.cuda.synchronize()
            kc.finalise_launch(thr, counts_ptr=u32.data_ptr())
            _check(tuple(x.copy() for x in kc.results()), want, special, thr, wrapped)

        # the same counters through the live buffer and the reduction's snapshot
        thr = THRESHOLDS[0]
        want = _oracle(orc, keys, variant, allele, counts, nv, n_children, thr)
        live = dist.counts_tensor(kc)
        live.copy_(u32)
        torch.cuda.synchronize()
        kc.reduce_push(thr)
        kc.reset_counts()
        kc.reduce_flush(thr)
        assert np.array_equal(kc.reduced_counts().astype(np.uint64), counts)
        _check(tuple(x.copy() for x in kc.results()), want, special, thr, _wrapped_calls(orc, want, n_children, thr))
