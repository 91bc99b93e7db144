"""Synthetic trios of the shapes BASELINE.json names (SURVEY.md §8d): a seeded random
genome, planted SNV / indel candidate DNMs, fixed-length reads at a target depth with
sequencing errors, N bases and a base-quality model.  Data generation only — nothing
here counts k-mers.

Two generators with the same model:
  * `make_trio_host`   — NumPy, decoded reads (ASCII + qualities), for parity tests and
                         the CPU baseline sample (`make_family_host`: the same for a family
                         of one mother, one father and several children);
  * `make_sample_device` — PyTorch on the GPU, emits the packed stream (2-bit bases +
                         1-bit flags + separators) directly in HBM for the bench.
"""
from dataclasses import dataclass, field

import numpy as np

ASCII = np.frombuffer(b"ACGT", dtype=np.uint8)
COMP_ASCII = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTN", b"TGCAN"):
    COMP_ASCII[_a] = _b


@dataclass
class Variant:
    pos: int      # 0-based position of REF's first base in the genome
    ref: str
    alt: str
    inherited: bool = False  # also carried by the mother (should NOT be called de novo)
    # family generator: the child that owns the variant, and the children that carry it (the
    # trio generators: child 0 carries every variant)
    owner: int = 0
    carriers: frozenset = frozenset({0})


@dataclass
class Trio:
    k: int
    genome: np.ndarray  # uint8 ASCII
    variants: list
    reads: dict = field(default_factory=dict)  # sample -> (seq uint8, qual uint8, offsets uint64)
    # sample -> (lo, hi) uint64: each read's true alignment interval [lo, hi) in genome coordinates
    loci: dict = field(default_factory=dict)
    paralogs: list = field(default_factory=list)  # indices of the variants given a paralog copy
    n_children: int = 1  # reads / loci of child c are under sample child_sample(c)

    def variant_tuples(self):
        """(left flank, ref, alt, right flank) per variant, flanks k-1 long (shorter at ends)."""
        g = self.genome
        out = []
        for v in self.variants:
            lo = max(0, v.pos - (self.k - 1))
            end = v.pos + len(v.ref)
            out.append((g[lo:v.pos].tobytes().decode(), v.ref, v.alt,
                        g[end:end + self.k - 1].tobytes().decode()))
        return out


def make_genome(n: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return ASCII[rng.integers(0, 4, size=n, dtype=np.uint8)]


def plant_variants(genome: np.ndarray, n_variants: int, k: int, seed: int,
                   indel_frac: float = 0.0, inherited_frac: float = 0.1,
                   max_indel: int = 8) -> list:
    """Variants on a regular grid with jitter, at least 2k apart, away from the ends."""
    rng = np.random.default_rng(seed)
    n = len(genome)
    margin = 4 * k
    if n_variants == 0:
        return []
    step = (n - 2 * margin) // n_variants
    if step < 3 * k:
        raise ValueError("genome too short for this many variants")
    out = []
    for i in range(n_variants):
        pos = margin + i * step + int(rng.integers(0, step - 2 * k - max_indel))
        ref_base = chr(genome[pos])
        r = rng.random()
        if r < indel_frac / 2:  # insertion after the anchor base
            ins = "".join("ACGT"[b] for b in rng.integers(0, 4, size=int(rng.integers(1, max_indel + 1))))
            ref, alt = ref_base, ref_base + ins
        elif r < indel_frac:    # deletion of the bases after the anchor
            dl = int(rng.integers(1, max_indel + 1))
            ref, alt = genome[pos:pos + 1 + dl].tobytes().decode(), ref_base
        else:
            alt_base = "ACGT"[(("ACGT".index(ref_base)) + int(rng.integers(1, 4))) % 4]
            ref, alt = ref_base, alt_base
        out.append(Variant(pos, ref, alt, inherited=bool(rng.random() < inherited_frac)))
    return out


def apply_variants(genome: np.ndarray, variants) -> np.ndarray:
    """The alternate haplotype: genome with every given variant applied."""
    parts, cur = [], 0
    for v in sorted(variants, key=lambda x: x.pos):
        parts.append(genome[cur:v.pos])
        parts.append(np.frombuffer(v.alt.encode(), dtype=np.uint8))
        cur = v.pos + len(v.ref)
    parts.append(genome[cur:])
    return np.concatenate(parts)


def hap_ref_positions(genome: np.ndarray, variants) -> np.ndarray:
    """For every base of apply_variants(genome, variants): the genome position it aligns to.
    ALT base i of a variant at pos maps to pos + min(i, len(REF) - 1): substituted bases to
    themselves, inserted bases to their anchor, and a deletion's anchor to itself."""
    parts, cur = [], 0
    for v in sorted(variants, key=lambda x: x.pos):
        parts.append(np.arange(cur, v.pos, dtype=np.int64))
        parts.append(v.pos + np.minimum(np.arange(len(v.alt)), len(v.ref) - 1))
        cur = v.pos + len(v.ref)
    parts.append(np.arange(cur, len(genome), dtype=np.int64))
    return np.concatenate(parts)


def read_loci(refpos, hap_of, starts, lens):
    """Alignment intervals [lo, hi) in genome coordinates of reads drawn from haplotypes whose
    bases align to refpos[h] (hap_ref_positions; None = the genome itself): the aligned
    positions of the read's first and last base.  An empty read gets [lo, lo)."""
    hap_of = np.asarray(hap_of, dtype=np.int64)
    starts = np.asarray(starts, dtype=np.int64)
    lens = np.asarray(lens, dtype=np.int64)
    lo = np.zeros(len(starts), dtype=np.int64)
    hi = np.zeros(len(starts), dtype=np.int64)
    last = starts + np.maximum(lens, 1) - 1
    for h, rp in enumerate(refpos):
        sel = hap_of == h
        lo[sel] = starts[sel] if rp is None else rp[starts[sel]]
        hi[sel] = (last[sel] if rp is None else rp[last[sel]]) + 1
    hi = np.where(lens > 0, hi, lo)
    return lo.astype(np.uint64), hi.astype(np.uint64)


def sample_reads(haps, n_reads: int, read_len: int, seed: int, err_rate: float = 0.002,
                 n_rate: float = 0.0005, lowq_frac: float = 0.03, rc_frac: float = 0.5,
                 ragged: bool = False, return_meta: bool = False):
    """Reads drawn uniformly from the given haplotypes (equal weight).  Returns
    (seq ASCII uint8, qual uint8, offsets uint64[n_reads+1]); with return_meta also
    (haplotype of each read, its start on that haplotype)."""
    rng = np.random.default_rng(seed)
    hap_of = rng.integers(0, len(haps), size=n_reads)
    lens = np.full(n_reads, read_len, dtype=np.int64)
    if ragged:
        lens = rng.integers(1, read_len + 1, size=n_reads)
    offsets = np.zeros(n_reads + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(lens)
    total = int(offsets[-1])
    seq = np.empty(total, dtype=np.uint8)
    all_starts = np.zeros(n_reads, dtype=np.int64)
    for h, hap in enumerate(haps):
        idx = np.nonzero(hap_of == h)[0]
        if len(idx) == 0:
            continue
        starts = rng.integers(0, len(hap) - read_len + 1, size=len(idx))
        all_starts[idx] = starts
        if not ragged:  # fixed length: one gather
            seq.reshape(n_reads, read_len)[idx] = hap[starts[:, None] + np.arange(read_len)[None, :]]
            continue
        for r, s in zip(idx, starts):
            seq[int(offsets[r]):int(offsets[r + 1])] = hap[s:s + int(lens[r])]
    # sequencing errors: substitute with a different base
    err = rng.random(total) < err_rate
    if err.any():
        code = np.searchsorted(ASCII, seq[err])  # ASCII is sorted A<C<G<T
        seq[err] = ASCII[(code + rng.integers(1, 4, size=int(err.sum()))) % 4]
    # reverse-complement a fraction of reads (reads from either strand)
    flip = rng.random(n_reads) < rc_frac
    if not ragged:
        m = seq.reshape(n_reads, read_len)
        m[flip] = COMP_ASCII[m[flip][:, ::-1]]
    else:
        for r in np.nonzero(flip)[0]:
            a, b = int(offsets[r]), int(offsets[r + 1])
            seq[a:b] = COMP_ASCII[seq[a:b][::-1]]
    seq[rng.random(total) < n_rate] = ord("N")
    qual = rng.integers(25, 41, size=total).astype(np.uint8)
    low = rng.random(total) < lowq_frac
    qual[low] = rng.integers(2, 20, size=int(low.sum())).astype(np.uint8)
    if return_meta:
        return seq, qual, offsets, (hap_of, all_starts)
    return seq, qual, offsets


def plant_paralogs(genome: np.ndarray, variants, k: int, which, seed: int, spacer: int = 20_000):
    """Append to the genome, `spacer` random bases past its end (so far from every candidate
    window), one copy of the 2k - 1 bases around each variant in `which` carrying its ALT
    allele, the copies `spacer` apart.  Every sample then holds that variant's alt k-mers at a
    second locus, as with a paralog or a segmental duplication."""
    rng = np.random.default_rng(seed)
    parts = [genome]
    for i in which:
        v = variants[i]
        end = v.pos + len(v.ref)
        parts.append(make_genome(spacer, int(rng.integers(1 << 30))))
        parts.append(genome[max(0, v.pos - (k - 1)):v.pos])
        parts.append(np.frombuffer(v.alt.encode(), dtype=np.uint8))
        parts.append(genome[end:end + k - 1])
    parts.append(make_genome(spacer, int(rng.integers(1 << 30))))
    return np.concatenate(parts)


def make_trio_host(genome_len: int, depth: float, n_variants: int, k: int, seed: int = 1,
                   read_len: int = 150, indel_frac: float = 0.0, ragged: bool = False,
                   paralog_frac: float = 0.0, **read_kw) -> Trio:
    """Child is heterozygous for every variant; the mother also carries the
    `inherited` ones; the father carries none.  trio.loci holds every read's true alignment
    interval.  paralog_frac: that fraction of the de novo (not inherited) variants gets an
    ALT-carrying copy far away (plant_paralogs; trio.paralogs lists them)."""
    genome = make_genome(genome_len, seed)
    variants = plant_variants(genome, n_variants, k, seed + 1, indel_frac=indel_frac)
    paralogs = []
    if paralog_frac > 0:
        rng = np.random.default_rng(seed + 3)
        denovo = [i for i, v in enumerate(variants) if not v.inherited]
        paralogs = sorted(rng.choice(denovo, size=max(1, int(round(paralog_frac * len(denovo)))),
                                     replace=False).tolist())
        genome = plant_paralogs(genome, variants, k, paralogs, seed + 4)
    child_alt = apply_variants(genome, variants)
    mother_var = [v for v in variants if v.inherited]
    mother_alt = apply_variants(genome, mother_var)
    n_reads = int(len(genome) * depth / read_len)
    trio = Trio(k, genome, variants, paralogs=paralogs)
    refpos = {0: [None, hap_ref_positions(genome, variants)],
              1: [None, hap_ref_positions(genome, mother_var)], 2: [None, None]}
    for smp, haps in enumerate([[genome, child_alt], [genome, mother_alt], [genome, genome]]):
        seq, qual, off, (hap_of, starts) = sample_reads(haps, n_reads, read_len, seed + 10 + smp, ragged=ragged,
                                                        return_meta=True, **read_kw)
        trio.reads[smp] = (seq, qual, off)
        trio.loci[smp] = read_loci(refpos[smp], hap_of, starts, np.diff(off).astype(np.int64))
    return trio


def child_sample(c: int) -> int:
    """Sample index of child c of a family (DKB_CHILD_SAMPLE in include/dkb.h): 0 for c == 0,
    else 2 + c.  (Kept here, not imported from the api: generating data loads no library.)"""
    return 0 if c == 0 else c + 2


def make_family_host(genome_len: int, depth: float, n_variants: int, k: int, n_children: int, seed: int = 1,
                     shared_frac: float = 0.2, inherited_frac: float = 0.2, indel_frac: float = 0.0,
                     paralog_frac: float = 0.0, read_len: int = 150, ragged: bool = False, **read_kw) -> Trio:
    """A family: mother (sample 1), father (sample 2) and n_children children (sample
    child_sample(c)), reads and loci keyed by sample index.  Variant i is owned by child
    i % n_children; each is, drawn independently:
      * inherited (inherited_frac): the mother carries it, each child with probability 1/2;
      * shared de novo (shared_frac, two children or more): the owner and one other child carry
        it, neither parent does (gonadal mosaicism in a parent);
      * de novo otherwise: only the owner carries it.
    Every child carrying a variant is heterozygous for it.  paralog_frac: that fraction of the
    variants not inherited gets an ALT-carrying copy far away (plant_paralogs)."""
    genome = make_genome(genome_len, seed)
    variants = plant_variants(genome, n_variants, k, seed + 1, indel_frac=indel_frac, inherited_frac=0.0)
    rng = np.random.default_rng(seed + 2)
    for i, v in enumerate(variants):
        v.owner = i % n_children
        r = rng.random()
        if r < inherited_frac:
            v.inherited = True
            v.carriers = frozenset(int(c) for c in np.nonzero(rng.random(n_children) < 0.5)[0])
        elif r < inherited_frac + shared_frac and n_children > 1:
            other = (v.owner + 1 + int(rng.integers(0, n_children - 1))) % n_children
            v.carriers = frozenset({v.owner, other})
        else:
            v.carriers = frozenset({v.owner})
    paralogs = []
    if paralog_frac > 0:
        prng = np.random.default_rng(seed + 3)
        denovo = [i for i, v in enumerate(variants) if not v.inherited]
        paralogs = sorted(prng.choice(denovo, size=max(1, int(round(paralog_frac * len(denovo)))),
                                      replace=False).tolist())
        genome = plant_paralogs(genome, variants, k, paralogs, seed + 4)
    carried = {1: [v for v in variants if v.inherited], 2: []}
    for c in range(n_children):
        carried[child_sample(c)] = [v for v in variants if c in v.carriers]
    n_reads = int(len(genome) * depth / read_len)
    fam = Trio(k, genome, variants, paralogs=paralogs, n_children=n_children)
    for smp in sorted(carried):
        alt = apply_variants(genome, carried[smp])
        refpos = [None, hap_ref_positions(genome, carried[smp])]
        seq, qual, off, (hap_of, starts) = sample_reads([genome, alt], n_reads, read_len, seed + 10 + smp,
                                                        ragged=ragged, return_meta=True, **read_kw)
        fam.reads[smp] = (seq, qual, off)
        fam.loci[smp] = read_loci(refpos, hap_of, starts, np.diff(off).astype(np.int64))
    return fam


# Locus classes and sexes of include/dkb.h (DKB_LOCUS_*, DKB_SEX_*)
LOCUS_AUTOSOMAL, LOCUS_X, LOCUS_Y, LOCUS_MATERNAL = 0, 1, 2, 3
SEX_UNKNOWN, SEX_MALE, SEX_FEMALE = 0, 1, 2

# The planted scenarios of make_sexed_family_host: name -> (locus class, the call byte the
# inheritance rule gives a son, the byte it gives a daughter) at error-free reads and the
# default thresholds (3, 2, 0, 1).  A parent whose one copy of X or MT carries the alt has no
# ref hits there, so where that parent's clauses apply the byte has DKB_CALL_PARENT_UNCOVERED.
SEXED_SCENARIOS = {
    # the son's X comes from his mother: his alt is de novo although his father carries it
    "x_denovo_carrier_father": (LOCUS_X, 0x01, 0x18),
    # the daughter inherits her father's X and its alt; the son does not carry it
    "x_inherited_paternal": (LOCUS_X, 0x02, 0x18),
    # a son's de novo on Y; a daughter has no Y
    "y_denovo": (LOCUS_Y, 0x01, 0x22),
    # a child's MT de novo at a site where the father's own MT carries the alt
    "mt_denovo_carrier_father": (LOCUS_MATERNAL, 0x01, 0x01),
    # every child inherits the mother's MT alt, which the father's own MT carries too
    "mt_inherited_maternal": (LOCUS_MATERNAL, 0x14, 0x14),
    # autosomal controls: de novo in every child, and inherited from the mother by every child
    "autosomal_denovo": (LOCUS_AUTOSOMAL, 0x01, 0x01),
    "autosomal_inherited": (LOCUS_AUTOSOMAL, 0x04, 0x04),
}


@dataclass
class SexedFamily(Trio):
    classes: np.ndarray = None  # uint8 locus class per variant (LOCUS_*)
    sexes: list = None          # sex of child c (SEX_MALE / SEX_FEMALE)
    scenarios: list = None      # SEXED_SCENARIOS name of each variant
    segments: dict = None       # locus class -> [start, end) of its segment in the genome


def make_sexed_family_host(sexes, k: int, seed: int = 1, depth: float = 20, per_scenario: int = 3,
                           seg_len=(60_000, 40_000, 20_000, 16_000), read_len: int = 150,
                           **read_kw) -> SexedFamily:
    """A family whose samples hold an autosome, X, Y and mitochondrial (MT) segment at the copy
    numbers of their sex: mother (sample 1) autosome x2, X x2, her own MT; father (sample 2)
    autosome x2, X x1, Y x1, his own MT; child c (sample child_sample(c)) of sexes[c] the
    autosome x2, the mother's first X, and the father's X (daughter) or Y (son), and the
    mother's MT.  Depth is per copy, so hemizygous segments come out at half the depth.  The
    segments lie back to back in one genome (fam.segments), and read loci are in its
    coordinates.  per_scenario SNVs of every SEXED_SCENARIOS scenario are planted, each 3k or
    more from the next; fam.scenarios names each variant's, fam.classes gives its locus class."""
    sexes = [int(s) for s in sexes]
    assert sexes and all(s in (SEX_MALE, SEX_FEMALE) for s in sexes)
    rng = np.random.default_rng(seed)
    order = (LOCUS_AUTOSOMAL, LOCUS_X, LOCUS_Y, LOCUS_MATERNAL)
    genome = make_genome(sum(seg_len), seed)
    segments, s0 = {}, 0
    for cls, n in zip(order, seg_len):
        segments[cls] = (s0, s0 + n)
        s0 += n
    # SNVs on an even grid inside their segment, away from its ends
    by_cls = {c: [name for name, sc in SEXED_SCENARIOS.items() if sc[0] == c] for c in order}
    variants, scen = [], []
    for cls in order:
        names = [nm for nm in by_cls[cls] for _ in range(per_scenario)]
        lo, hi = segments[cls]
        step = (hi - lo - 8 * k) // max(len(names), 1)
        assert step >= 3 * k, "segment too short for its scenarios"
        for i, nm in enumerate(names):
            pos = lo + 4 * k + i * step + int(rng.integers(0, step - 2 * k))
            ref = chr(genome[pos])
            alt = "ACGT"[("ACGT".index(ref) + int(rng.integers(1, 4))) % 4]
            variants.append(Variant(pos, ref, alt))
            scen.append(nm)

    def alts(*names):
        """{pos: alt base} of every variant of the named scenarios"""
        return {v.pos: v.alt for v, nm in zip(variants, scen) if nm in names}

    # copies: (locus class, {pos: base})
    mat_a = (LOCUS_AUTOSOMAL, alts("autosomal_inherited"))
    mat_x = (LOCUS_X, {})
    mat_mt = (LOCUS_MATERNAL, alts("mt_inherited_maternal"))
    pat_x = (LOCUS_X, alts("x_denovo_carrier_father", "x_inherited_paternal"))
    pat_y = (LOCUS_Y, {})
    copies = {
        1: [mat_a, (LOCUS_AUTOSOMAL, {}), mat_x, (LOCUS_X, {}), mat_mt],
        2: [(LOCUS_AUTOSOMAL, {}), (LOCUS_AUTOSOMAL, {}), pat_x, pat_y,
            (LOCUS_MATERNAL, alts("mt_denovo_carrier_father", "mt_inherited_maternal"))],
    }
    for c, sex in enumerate(sexes):
        child = [mat_a, (LOCUS_AUTOSOMAL, alts("autosomal_denovo")),
                 (LOCUS_MATERNAL, {**mat_mt[1], **alts("mt_denovo_carrier_father")})]
        if sex == SEX_MALE:
            child += [(LOCUS_X, alts("x_denovo_carrier_father")), (LOCUS_Y, alts("y_denovo"))]
        else:
            child += [mat_x, pat_x]
        copies[child_sample(c)] = child
    fam = SexedFamily(k, genome, variants, n_children=len(sexes), classes=np.array(
        [SEXED_SCENARIOS[nm][0] for nm in scen], dtype=np.uint8), sexes=sexes, scenarios=scen, segments=segments)
    for smp in sorted(copies):
        seqs, quals, lens, los = [], [], [], []
        for j, cls in enumerate(order):
            lo, hi = segments[cls]
            haps = []
            for ccls, edits in copies[smp]:
                if ccls != cls:
                    continue
                h = genome[lo:hi].copy()
                for p, b in edits.items():
                    h[p - lo] = ord(b)
                haps.append(h)
            if not haps:
                continue
            n_reads = int(round((hi - lo) * depth * len(haps) / read_len))
            seq, qual, off, (hap_of, starts) = sample_reads(haps, n_reads, read_len, seed + 10 + 4 * smp + j,
                                                            return_meta=True, **read_kw)
            seqs.append(seq)
            quals.append(qual)
            lens.append(np.diff(off).astype(np.int64))
            los.append(starts + lo)
        lens = np.concatenate(lens)
        off = np.zeros(len(lens) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        fam.reads[smp] = (np.concatenate(seqs), np.concatenate(quals), off)
        lo = np.concatenate(los)
        fam.loci[smp] = (lo.astype(np.uint64), (lo + lens).astype(np.uint64))
    return fam


# ---------------------------------------------------------------------------------------
# GPU generator: packed streams built in HBM (bench workload; no host copy of the reads)
# ---------------------------------------------------------------------------------------
def make_sample_device(haps_codes, n_reads: int, read_len: int, seed: int, device,
                       err_rate: float = 0.002, n_rate: float = 0.0005, lowq_frac: float = 0.03,
                       rc_frac: float = 0.5, chunk_reads: int = 1 << 20, return_meta: bool = False):
    """haps_codes: list of uint8 CUDA tensors of base codes 0..3 (one per haplotype).
    Returns (bases2 int32 tensor, mask1 int32 tensor, n_positions, n_bases) in the layout
    of include/dkb.h.  Same read model as `sample_reads`; low-quality and N bases only
    clear the flag (what the host packer would emit)."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    stride = read_len + 1  # one separator per read
    n_pos = n_reads * stride
    bw = (n_pos + 63) // 64 * 4
    mw = (n_pos + 127) // 128 * 4
    bases2 = torch.zeros(bw, dtype=torch.int32, device=device)
    mask1 = torch.zeros(mw, dtype=torch.int32, device=device)
    # chunks must cover whole 128-position groups: chunk_reads * stride % 128 == 0
    chunk_reads = max(128, chunk_reads // 128 * 128)
    ar = torch.arange(read_len, device=device)
    sh2 = (2 * torch.arange(16, device=device, dtype=torch.int64))
    sh1 = torch.arange(32, device=device, dtype=torch.int64)
    meta_h, meta_s = [], []
    for r0 in range(0, n_reads, chunk_reads):
        nr = min(chunk_reads, n_reads - r0)
        codes = torch.zeros((nr, stride), dtype=torch.uint8, device=device)
        valid = torch.zeros((nr, stride), dtype=torch.bool, device=device)
        hap_of = torch.randint(0, len(haps_codes), (nr,), generator=g, device=device)
        body = torch.empty((nr, read_len), dtype=torch.uint8, device=device)
        all_starts = torch.zeros((nr,), dtype=torch.int64, device=device)
        for h, hap in enumerate(haps_codes):
            sel = (hap_of == h).nonzero().squeeze(1)
            if sel.numel() == 0:
                continue
            starts = torch.randint(0, hap.numel() - read_len + 1, (sel.numel(),), generator=g,
                                   device=device)
            body[sel] = hap[starts[:, None] + ar[None, :]]
            all_starts[sel] = starts
        if return_meta:
            meta_h.append(hap_of)
            meta_s.append(all_starts)
        err = torch.rand((nr, read_len), generator=g, device=device) < err_rate
        bump = torch.randint(1, 4, (nr, read_len), generator=g, device=device, dtype=torch.uint8)
        body = torch.where(err, (body + bump) & 3, body)
        flip = torch.rand((nr,), generator=g, device=device) < rc_frac
        body = torch.where(flip[:, None], 3 - body.flip(1), body)
        ok = torch.rand((nr, read_len), generator=g, device=device) >= (n_rate + lowq_frac)
        codes[:, :read_len] = torch.where(ok, body, torch.zeros_like(body))
        valid[:, :read_len] = ok
        flat_c = codes.reshape(-1)
        flat_v = valid.reshape(-1)
        p0 = r0 * stride
        pad = (-flat_c.numel()) % 128
        if pad:
            flat_c = torch.cat([flat_c, flat_c.new_zeros(pad)])
            flat_v = torch.cat([flat_v, flat_v.new_zeros(pad)])
        wb = (flat_c.reshape(-1, 16).to(torch.int64) << sh2).sum(1)
        wm = (flat_v.reshape(-1, 32).to(torch.int64) << sh1).sum(1)
        # int64 -> wrap into int32 bit patterns
        wb = torch.where(wb >= 2 ** 31, wb - 2 ** 32, wb).to(torch.int32)
        wm = torch.where(wm >= 2 ** 31, wm - 2 ** 32, wm).to(torch.int32)
        assert p0 % 128 == 0
        bases2[p0 // 16: p0 // 16 + wb.numel()] = wb[: bases2.numel() - p0 // 16]
        mask1[p0 // 32: p0 // 32 + wm.numel()] = wm[: mask1.numel() - p0 // 32]
    if return_meta:
        return bases2, mask1, n_pos, n_reads * read_len, (torch.cat(meta_h), torch.cat(meta_s))
    return bases2, mask1, n_pos, n_reads * read_len


def device_read_loci(meta, refpos, read_len: int):
    """The loci of make_sample_device's reads from its return_meta output: (offsets, lo, hi)
    uint64 host arrays for dkb_batch_set_loci.  refpos[h]: hap_ref_positions of haplotype h
    (None = the genome itself)."""
    hap_of, starts = (t.cpu().numpy() for t in meta)
    n = len(starts)
    offsets = np.arange(n + 1, dtype=np.uint64) * np.uint64(read_len)
    lo, hi = read_loci(refpos, hap_of, starts, np.full(n, read_len, dtype=np.int64))
    return offsets, lo, hi
