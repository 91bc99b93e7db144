// dkb_pack.cuh — kernel 0: device-side read packer (widening row f1 of DESIGN.md §0).
// Same output as the host packer dkb_pack_reads, bit for bit, from decoded reads left in
// the form the BAM layer already holds: bases as ASCII or as BAM's 4-bit codes, one
// quality byte per base.  One thread builds 32 stream positions (two base words, one
// mask word), so no output word is shared between threads.  Both kernels of this file take
// every batch of one submit (up to MAX_SEGMENTS) in one launch.
#pragma once
#include "dkb_device.cuh"

namespace dkb {

// BAM 4-bit code -> 2-bit code (A=1 C=2 G=4 T=8), 4 = not a plain base
__device__ __forceinline__ uint32_t nib_to_code(uint32_t n) {
  return n == 1 ? 0u : n == 2 ? 1u : n == 4 ? 2u : n == 8 ? 3u : 4u;
}
__device__ __forceinline__ uint32_t ascii_to_code(uint32_t c) {
  c &= 0xDFu;  // fold case
  return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
}

// One batch of a k_pack launch: its reads in the staging slot, and where its stream goes.
struct PackSegment {
  const uint8_t *seq;        // ASCII bases, or 4-bit codes (high nibble first, BAM order)
  const uint8_t *qual;       // may be null
  const uint64_t *offsets;   // [n_reads + 1] base offsets of the reads in seq/qual (ASCII form)
  const uint64_t *nib_start; // [n_reads] byte offset of each read's first nibble pair (4-bit form)
  uint32_t *bases2;
  uint32_t *mask1;
  uint64_t m_begin;          // first mask word of the batch in the launch's global numbering
  uint64_t n_pos;
  uint32_t n_reads;
  uint32_t n_bwords, n_mwords;  // output sizes (dkb_stream_*_words)
};

// The batches of one submit (up to MAX_SEGMENTS), packed by one launch: segment i owns the
// global mask words [seg[i].m_begin, seg[i].m_begin + seg[i].n_mwords).
struct PackParams {
  PackSegment seg[MAX_SEGMENTS];
  uint32_t n_seg;
  uint64_t n_mwords;  // all segments
  int min_baseq;
  int four_bit;
};

__global__ void k_pack(const PackParams Q) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // global mask word index
  if (g >= Q.n_mwords) return;
  uint32_t sg = 0;
#pragma unroll
  for (uint32_t j = 1; j < MAX_SEGMENTS; j++)
    if (j < Q.n_seg && g >= Q.seg[j].m_begin) sg = j;
  const PackSegment &S = Q.seg[sg];
  const uint64_t m = g - S.m_begin;  // mask word inside the batch
  const uint64_t p0 = m * 32;
  uint32_t b0 = 0, b1 = 0, mk = 0;
  if (p0 < S.n_pos && S.n_reads) {
    // read r starts at stream position offsets[r] - offsets[0] + r; find the last start <= p0
    const uint64_t o0 = S.offsets[0];
    uint32_t lo = 0, hi = S.n_reads;
    while (hi - lo > 1) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (S.offsets[mid] - o0 + mid <= p0) lo = mid; else hi = mid;
    }
    uint32_t r = lo;
    uint64_t start = S.offsets[r] - o0 + r;
    uint64_t len = S.offsets[r + 1] - S.offsets[r];
    uint64_t i = p0 - start;  // offset inside read r; i == len is the separator
    for (uint32_t t = 0; t < 32 && p0 + t < S.n_pos; t++) {
      if (i < len) {
        uint32_t c;
        if (Q.four_bit) {
          const uint32_t byte = S.seq[S.nib_start[r] + (i >> 1)];
          c = nib_to_code((i & 1) ? (byte & 15u) : (byte >> 4));
        } else {
          c = ascii_to_code(S.seq[S.offsets[r] - o0 + i]);  // device copies start at the batch's first base
        }
        const bool ok = c < 4 && (S.qual == nullptr || (int)S.qual[S.offsets[r] - o0 + i] >= Q.min_baseq);
        if (ok) {
          mk |= 1u << t;
          if (t < 16) b0 |= c << (2 * t); else b1 |= c << (2 * (t - 16));
        }
        i++;
      } else {  // separator, then the next read
        r++;
        i = 0;
        if (r < S.n_reads) len = S.offsets[r + 1] - S.offsets[r]; else len = 0;
      }
    }
  }
  if (2 * m < S.n_bwords) S.bases2[2 * m] = b0;
  if (2 * m + 1 < S.n_bwords) S.bases2[2 * m + 1] = b1;
  S.mask1[m] = mk;
}

// ---- zero list -> dense flags --------------------------------------------------------
// The flags of a stream can travel as a ZERO LIST instead of one bit per position (format:
// include/dkb.h, dkb_mask_to_zero_list): per block of ZL_BLOCK positions a byte string "skip g
// usable positions, then one unusable one" (255 = skip 255, no zero), or the block's plain bits
// when that is shorter.  One warp expands one block into its 64 mask words.
constexpr uint32_t ZL_BLOCK = 2048;           // positions per block = 64 mask words
constexpr uint32_t ZL_RAW_BIT = 0x80000000u;  // in zoff[b]: the block is stored as plain bits (256 bytes)

// One batch of a k_expand_zero_list launch: its zero list in the staging slot and its output
// flags.  Segment i owns the launch's global blocks [b_begin, b_begin + n_blocks).
struct ZeroListSegment {
  const uint32_t *zoff;
  const uint8_t *zbytes;
  uint32_t *mask1;
  uint32_t b_begin, n_blocks, n_mwords;
};
struct ZeroListParams {
  ZeroListSegment seg[MAX_SEGMENTS];
  uint32_t n_seg;
  uint32_t n_blocks;  // all segments
};

__global__ void k_expand_zero_list(const ZeroListParams Z) {
  __shared__ uint32_t sm[8][64];  // blockDim = 256: 8 warps
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * 8 + warp;  // global block
  if (g >= Z.n_blocks) return;
  uint32_t sg = 0;
#pragma unroll
  for (uint32_t j = 1; j < MAX_SEGMENTS; j++)
    if (j < Z.n_seg && g >= Z.seg[j].b_begin) sg = j;
  const ZeroListSegment &S = Z.seg[sg];
  const uint32_t b = g - S.b_begin;  // block inside the batch
  uint32_t *w = sm[warp];
  const uint32_t o0 = S.zoff[b], o1 = S.zoff[b + 1] & ~ZL_RAW_BIT;
  const uint8_t *src = S.zbytes + (o0 & ~ZL_RAW_BIT);
  if (o0 & ZL_RAW_BIT) {  // plain bits, little-endian words
    for (int i = lane; i < 64; i += 32) {
      uint32_t v = 0;
      for (int k = 0; k < 4; k++) v |= (uint32_t)src[4 * i + k] << (8 * k);
      w[i] = v;
    }
  } else {
    w[lane] = 0xFFFFFFFFu;
    w[lane + 32] = 0xFFFFFFFFu;
    __syncwarp();
    const uint32_t n = o1 - (o0 & ~ZL_RAW_BIT);
    uint32_t carry = 0;  // positions consumed so far
    for (uint32_t i0 = 0; i0 < n; i0 += 32) {
      const uint32_t i = i0 + lane;
      const uint32_t v = i < n ? src[i] : 255u;
      const uint32_t adv = i < n ? (v == 255u ? 255u : v + 1u) : 0u;
      uint32_t incl = adv;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL_MASK, incl, o);
        if (lane >= o) incl += t;
      }
      if (i < n && v != 255u) {
        const uint32_t pos = carry + incl - 1u;  // the zero position, inside the block
        if (pos < ZL_BLOCK) atomicAnd(&w[pos >> 5], ~(1u << (pos & 31)));
      }
      carry += __shfl_sync(FULL_MASK, incl, 31);
    }
  }
  __syncwarp();
  for (int i = lane; i < 64; i += 32) {
    const size_t m = (size_t)b * 64 + i;
    if (m < S.n_mwords) S.mask1[m] = w[i];
  }
}

}  // namespace dkb
