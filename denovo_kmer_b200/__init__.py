"""denovo_kmer_b200 — B200-native hot path of jlanej/denovo_kmer (k-mer extraction from
child/parent reads + membership counting against candidate alleles' spanning k-mers +
de novo support thresholds) behind a C ABI (include/dkb.h, libdkb.so).

The CUDA library is the only compute path: importing works without it (so the build
step can import the package), but any call raises ImportError until it is built, and
DKB_ENODEV without a B200.
"""
from .api import (ALT, CALL_CHILD_LOW, CALL_DENOVO, CALL_FATHER_ALT, CALL_MOTHER_ALT,  # noqa: F401
                  CALL_NO_COPY, CALL_PARENT_UNCOVERED, CHILD, DEFAULT_MIN_BASEQ, DEFAULT_THRESHOLDS, FATHER,
                  LOCUS_AUTOSOMAL, LOCUS_MATERNAL, LOCUS_X, LOCUS_Y, SEX_FEMALE, SEX_MALE, SEX_UNKNOWN,
                  MAX_CHILDREN, MOTHER, REF, KmerCounter, KmerEntries, ReadLoci, ReadStream, child_sample, kmer_canonical,
                  comm_unique_id, kmer_encode, mask_to_zero_list, kmer_revcomp, pack_reads, stream_words, variant_kmers)
from ._lib import DkbError  # noqa: F401

__version__ = "0.2.0"
