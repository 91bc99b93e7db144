"""Seeded adversarial inputs for the scan kernels: one trio of read batches plus read loci, made to
reach the paths random genomes rarely reach (tests/test_gpu_kernel_matrix.py runs every built
kernel on them; tests/test_adversarial_inputs.py asserts, on the CPU, that they still do):

  * dense, low-complexity reads (poly-A, dinucleotide, trinucleotide, >= 20 000 bases) and
    candidates with low-complexity flanks: every lookup of a macro tile hits the filter;
  * hundreds of copies of one alt-haplotype read: stage C's ring wraps, many hits per lane;
  * multi-owner keys: a multiallelic STR split into 40 biallelic records with identical flanks,
    and one candidate repeated 40 times as paralog copies;
  * a key-table chain that starts in the last bucket and wraps to bucket 0 (key_bucket mirrors
    the device function of the same name in dkb_device.cuh);
  * palindromes: an alt window that is its own reverse complement (even k), whose windows hold
    palindromic 14-mers at every interior offset;
  * stream edges: every batch starts on a candidate's alt window and ends on one, and the batch
    lengths n_pos are 0, +1, -1 and 6144 modulo 16 384;
  * reads of length k - 1, k and k + 1, an N every k-th base, low-quality runs;
  * loci: reads on their candidate's window, far away, or unmapped."""
from dataclasses import dataclass, field

import numpy as np

FLANK = 40
MIN_BQ = 20
PAD = 100
N_STR, N_PARALOG, N_WRAP_COPIES, N_DENSE = 40, 40, 4, 300
LOW_COMPLEXITY = ("A", "AC", "ACG")
LOW_COMPLEXITY_LEN = 20_000
RESIDUES = (0, 1, 16383, 6144)  # n_pos of the four batches modulo 16 384
FAR = 1 << 40
_COMP = str.maketrans("ACGT", "TGCA")
_CODE = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i


def revcomp(s):
    return s.translate(_COMP)[::-1]


def window_keys(seq, k):
    """Canonical keys (first base most significant) of every window of an ACGT string."""
    c = _CODE[np.frombuffer(seq.encode(), dtype=np.uint8)].astype(np.uint64)
    n = len(c) - k + 1
    if n <= 0:
        return np.zeros(0, dtype=np.uint64)
    fwd = np.zeros(n, dtype=np.uint64)
    rc = np.zeros(n, dtype=np.uint64)
    for j in range(k):
        fwd = (fwd << np.uint64(2)) | c[j:j + n]
        rc |= (np.uint64(3) - c[j:j + n]) << np.uint64(2 * j)
    return np.minimum(fwd, rc)


def key_bucket(keys, bucket_mask):
    """dkb_device.cuh key_bucket, over uint64 arrays."""
    keys = np.asarray(keys, dtype=np.uint64)
    m32 = np.uint64(0xFFFFFFFF)
    x = (keys & m32) ^ (((keys >> np.uint64(32)) * np.uint64(0x9E3779B1)) & m32)
    x = (x * np.uint64(0x85EBCA6B)) & m32
    x ^= x >> np.uint64(15)
    return x & np.uint64(bucket_mask)


def table_slots(n_entries):
    """Key-table slots of a table of n_entries (dkb_table_build: 8 per entry, a power of two)."""
    p = 1024
    while p < 8 * n_entries + 2:
        p <<= 1
    return p


def n_positions(off):
    return int(off[-1] - off[0]) + len(off) - 1


@dataclass
class Batch:
    sample: int
    seq: np.ndarray   # uint8 ASCII
    qual: np.ndarray  # uint8
    off: np.ndarray   # uint64, from 0
    lo: np.ndarray    # uint64 read loci
    hi: np.ndarray


@dataclass
class Input:
    k: int
    variants: list               # (left, ref, alt, right)
    pos: np.ndarray              # locus of each variant
    vlo: np.ndarray
    vhi: np.ndarray
    batches: list
    facts: dict = field(default_factory=dict)  # what the builder planted, for the precondition checks


def _rand(rng, n):
    return "".join("ACGT"[i] for i in rng.integers(0, 4, n))


def _snv(rng):
    left, right = _rand(rng, FLANK), _rand(rng, FLANK)
    ref = "ACGT"[rng.integers(0, 4)]
    return left, ref, "ACGT".replace(ref, "")[rng.integers(0, 3)], right


def build(dkb, k, seed=0):
    rng = np.random.default_rng(seed)
    variants, facts = [], {}
    facts["snv"] = list(range(16))
    variants += [_snv(rng) for _ in range(16)]
    lc = lambda u, n: (u * (n // len(u) + 1))[:n]  # noqa: E731
    facts["low_complexity"] = list(range(len(variants), len(variants) + 4))
    variants += [(lc("A", FLANK), "A", "C", lc("A", FLANK)), (lc("AC", FLANK), "A", "G", lc("CA", FLANK)),
                 (lc("ACG", FLANK), "ACG", "A", lc("ACG", FLANK)), (lc("T", FLANK), "T", "TTT", lc("T", FLANK))]
    # multiallelic STR: one ref, 40 alt lengths, identical flanks
    sl, sr = _rand(rng, FLANK), _rand(rng, FLANK)
    facts["str"] = list(range(len(variants), len(variants) + N_STR))
    variants += [(sl, "CA" * 10, "CA" * j, sr) for j in range(1, N_STR + 2) if j != 10]
    facts["paralog"] = list(range(len(variants), len(variants) + N_PARALOG))
    variants += [_snv(rng)] * N_PARALOG
    # palindrome: the alt haplotype holds X + rc(X), |X| = 15, with the alt base inside X
    x = _rand(rng, 15)
    ref = "ACGT".replace(x[14], "")[0]
    facts["palindrome"] = len(variants)
    facts["palindrome_window"] = x + revcomp(x)
    variants.append((_rand(rng, FLANK - 14) + x[:14], ref, x[14], revcomp(x) + _rand(rng, FLANK - 15)))

    # a candidate repeated N_WRAP_COPIES times with one alt key homed in the table's last bucket
    # (the table's size depends on the entry count: an SNV with random flanks has 2k entries)
    mask = table_slots(len(dkb.variant_kmers(variants, k)) + N_WRAP_COPIES * 2 * k) // 2 - 1
    while True:
        cand = _snv(rng)
        alt_hap = cand[0] + cand[2] + cand[3]
        keys = window_keys(alt_hap[FLANK - k + 1:FLANK + k], k)
        hit = np.nonzero(key_bucket(keys, mask) == mask)[0]
        if len(hit) and table_slots(len(dkb.variant_kmers(variants + [cand] * N_WRAP_COPIES, k))) // 2 - 1 == mask:
            break
    facts["wrap"] = list(range(len(variants), len(variants) + N_WRAP_COPIES))
    facts["wrap_key"] = int(keys[hit[0]])
    variants += [cand] * N_WRAP_COPIES

    pos = np.array([10_000 * (i + 1) for i in range(len(variants))], dtype=np.uint64)
    pos[facts["str"]] = pos[facts["str"][0]]
    vlo = pos - PAD
    vhi = pos + np.array([len(v[1]) for v in variants], dtype=np.uint64) + PAD

    def hap(i, allele):
        left, r, a, right = variants[i]
        return left + (a if allele else r) + right

    def from_hap(i, allele, a, b):
        """Read hap[a:b] of variant i with its locus."""
        lo = int(pos[i]) - FLANK + a
        return hap(i, allele)[a:b], lo, lo + (b - a)

    def cover(i, allele, rlen):
        h = hap(i, allele)
        a = int(rng.integers(max(0, FLANK + 1 - rlen), FLANK + 1))
        return from_hap(i, allele, a, min(len(h), a + rlen))

    uniq = facts["snv"] + facts["low_complexity"] + facts["str"] + facts["paralog"][:2] + [facts["palindrome"]] + \
        facts["wrap"][:1]
    reads = {0: [], 1: [], 2: []}
    for smp in range(3):
        for i in uniq:
            for _ in range(2):
                reads[smp].append(cover(i, 1 if smp == 0 or i in facts["paralog"] else 0, int(rng.integers(k + 2, 81))))
            reads[smp].append(cover(i, 0, int(rng.integers(k + 2, 81))))
        for u in LOW_COMPLEXITY:
            lo = int(pos[facts["low_complexity"][0]]) - LOW_COMPLEXITY_LEN // 2 if smp != 2 else FAR
            reads[smp].append((lc(u, LOW_COMPLEXITY_LEN + smp), lo, lo + LOW_COMPLEXITY_LEN))
        for d in (-1, 0, 1):  # k - 1, k, k + 1 bases ending just after the alt base
            reads[smp].append(from_hap(facts["snv"][1], 1, FLANK + 1 - (k + d), FLANK + 1))
        s, lo, hi = from_hap(facts["snv"][2], 1, 0, 2 * FLANK + 1)
        s = "".join("N" if j % k == k - 1 else c for j, c in enumerate(s + s))
        reads[smp].append((s, lo, hi))
    dense = from_hap(facts["snv"][0], 1, 0, 2 * FLANK + 1)
    reads[0] += [dense] * N_DENSE
    reads[1] += [from_hap(facts["palindrome"], 1, 0, 2 * FLANK + 1)] * 20
    facts["dense_read"] = dense[0]

    def batch(smp, rs, residue):
        order = rng.permutation(len(rs))
        rs = [rs[j] for j in order]
        # first read starts on an alt window, the last ends on one; a filler read sets n_pos
        first = from_hap(facts["snv"][3], 1, FLANK - k + 4, 2 * FLANK + 1)
        last = from_hap(facts["snv"][4], 1, 0, FLANK + 5)
        body = [first] + rs[:len(rs) // 2]
        tail = rs[len(rs) // 2:] + [last]
        n = sum(len(r[0]) + 1 for r in body + tail) + 1
        flen = 200 + (residue - (n + 200)) % 16384
        body.append((_rand(rng, flen), FAR, FAR + flen))
        rs = body + tail
        seq = "".join(r[0] for r in rs)
        off = np.zeros(len(rs) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(r[0]) for r in rs])
        qual = np.full(len(seq), 30, dtype=np.uint8)
        for r in rng.choice(len(rs), len(rs) // 10, replace=False):  # low-quality runs
            a = int(off[r]) + int(rng.integers(0, max(1, len(rs[r][0]) - 10)))
            qual[a:a + int(rng.integers(3, 11))] = 5
        lo = np.array([r[1] for r in rs], dtype=np.uint64)
        hi = np.array([r[2] for r in rs], dtype=np.uint64)
        moved = rng.random(len(rs)) < 0.2
        lo[moved] += np.uint64(FAR)
        hi[moved] += np.uint64(FAR)
        unmapped = rng.random(len(rs)) < 0.1
        hi[unmapped] = lo[unmapped]
        return Batch(smp, np.frombuffer(seq.encode(), dtype=np.uint8).copy(), qual, off, lo, hi)

    half = len(reads[0]) // 2
    parts = [(0, reads[0][:half]), (0, reads[0][half:]), (1, reads[1]), (2, reads[2])]
    batches = [batch(smp, rs, res) for (smp, rs), res in zip(parts, RESIDUES)]
    return Input(k, variants, pos, vlo, vhi, batches, facts)
