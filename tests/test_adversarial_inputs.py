"""CPU: the preconditions of the adversarial inputs (tests/adversarial.py) that the kernel matrix
(test_gpu_kernel_matrix.py) relies on, checked with the host library and the oracle, so that the
inputs cannot lose their teeth when the builder changes; and the builder's key_bucket mirror
against the library's own __host__ __device__ function, compiled for the host with nvcc."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import adversarial as adv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", params=[31, 30])
def built(request, dkb):
    k = request.param
    inp = adv.build(dkb, k, seed=k)
    return inp, dkb.variant_kmers(inp.variants, k)


def _live(orc, e):
    return orc.KmerSet(e.keys, e.variant, e.allele).live().astype(bool)


def test_multi_owner_keys_and_wrapping_chain(built, orc):
    inp, e = built
    live = _live(orc, e)
    _, owners = np.unique(e.keys[live], return_counts=True)
    assert owners.max() >= adv.N_STR and (owners >= adv.N_PARALOG).sum() >= 2 * inp.k
    mask = adv.table_slots(len(e)) // 2 - 1
    home = adv.key_bucket(e.keys[live], mask)
    assert (home == mask).sum() >= 3, "fewer than 3 live owners homed in the last bucket"
    assert ((e.keys[live] == inp.facts["wrap_key"]).sum()) == adv.N_WRAP_COPIES


def test_palindromes(built):
    inp, e = built
    k = inp.k
    key_set = set(e.keys.tolist())
    if k % 2 == 0:  # an alt window that is its own reverse complement is a key
        w = inp.facts["palindrome_window"]
        assert w == adv.revcomp(w) and int(adv.window_keys(w, k)[0]) in key_set
    # palindromic 14-mers at every interior offset 1..15 of some key window
    left, ref, alt, right = inp.variants[inp.facts["palindrome"]]
    hap = left + alt + right
    offs = set()
    for a in range(len(hap) - k + 1):
        if int(adv.window_keys(hap[a:a + k], k)[0]) not in key_set:
            continue
        offs |= {j for j in range(k - 13) if hap[a + j:a + j + 14] == adv.revcomp(hap[a + j:a + j + 14])}
    assert set(range(1, 16)) <= offs


def test_dense_reads_and_stream_edges(built, orc):
    inp, e = built
    k = inp.k
    key_set = set(e.keys.tolist())
    res = sorted(adv.n_positions(b.off) % 16384 for b in inp.batches)
    assert res == sorted(adv.RESIDUES) and [b.sample for b in inp.batches] == [0, 0, 1, 2]
    n_dense = long_lc = n_masked = 0
    lens = set()
    for b in inp.batches:
        reads = [b.seq[int(b.off[r]):int(b.off[r + 1])].tobytes().decode() for r in range(len(b.off) - 1)]
        first, last = reads[0], reads[-1]
        assert int(adv.window_keys(first[:k], k)[0]) in key_set  # seeds at stream positions < k - s
        assert int(adv.window_keys(last[-k:], k)[0]) in key_set  # neighbourhoods cut by n_pos
        n_dense += sum(r == inp.facts["dense_read"] for r in reads)
        long_lc += sum(len(r) >= adv.LOW_COMPLEXITY_LEN and r[:6] * 5 == r[:30]
                       for r in reads)
        lens |= {len(r) for r in reads}
        assert (b.qual < adv.MIN_BQ).any() and (b.hi <= b.lo).any() and (b.lo >= adv.FAR).any()
        n_masked += any("N" in r for r in reads)
    assert n_masked >= 3 and n_dense >= 200 and long_lc >= 3 * 3 and {k - 1, k, k + 1} <= lens
    # the dense read and the low-complexity flanks are counted by the oracle
    ks = orc.KmerSet(e.keys, e.variant, e.allele)
    c = ks.count_reads(np.frombuffer(inp.facts["dense_read"].encode(), dtype=np.uint8), None,
                       np.array([0, len(inp.facts["dense_read"])], dtype=np.uint64), k)
    assert c.sum() >= k
    lc_entries = np.isin(e.variant, inp.facts["low_complexity"])
    assert lc_entries.sum() > 0


def test_region_loci_cut_reads(built):
    inp, _ = built
    inside = outside = 0
    for b in inp.batches:
        for lo, hi in zip(b.lo.tolist(), b.hi.tolist()):
            hit = lo < hi and bool(((inp.vlo < hi) & (inp.vhi > lo)).any())
            inside += hit
            outside += not hit
    assert inside > 100 and outside > 10


def test_key_bucket_mirror_matches_device_header(tmp_path):
    """key_bucket of dkb_device.cuh compiled for the host by nvcc, against the Python mirror."""
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc) and not shutil.which(nvcc):
        pytest.skip("nvcc not found")
    src = tmp_path / "kb.cu"
    src.write_text('#include <cstdio>\n#include "dkb_device.cuh"\n'
                   "int main() { unsigned long long key; unsigned mask;\n"
                   '  while (scanf("%llu %u", &key, &mask) == 2) printf("%u\\n", dkb::key_bucket(key, mask));\n'
                   "  return 0; }\n")
    exe = tmp_path / "kb"
    subprocess.check_call([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                           "-I", os.path.join(ROOT, "denovo_kmer_b200", "csrc"), "-o", str(exe), str(src)],
                          cwd=tempfile.gettempdir())
    rng = np.random.default_rng(3)
    keys = np.concatenate([rng.integers(0, 1 << 62, 2000, dtype=np.uint64),
                           np.array([0, 1, (1 << 62) - 1, 0xFFFFFFFF, 1 << 32], dtype=np.uint64)])
    masks = (np.uint64(1) << rng.integers(9, 31, len(keys)).astype(np.uint64)) - np.uint64(1)
    out = subprocess.run([str(exe)], input="".join(f"{a} {m}\n" for a, m in zip(keys.tolist(), masks.tolist())),
                         capture_output=True, text=True, check=True).stdout.split()
    want = [int(adv.key_bucket(np.array([a], dtype=np.uint64), m)[0]) for a, m in zip(keys.tolist(), masks.tolist())]
    assert [int(x) for x in out] == want
