// K0 — genome ingest on the device.
// Replaces the in-memory products of get_genome_seq (pbsim.cpp:1032-1065): upper-cased sequence,
// per-base homopolymer length hp[] and the hpfreq[] histogram.  Device layout per sequence:
//   ascii : uint8[len]      upper-cased text (slow path and non-ACGT truth)
//   pk    : uint32[len/16]  2 bits per base, A=0 C=1 G=2 T=3 (complement = code ^ 3), base i at bits 2*(i&15)
//   hp4   : uint8[len/2]    4-bit homopolymer length (1..11, the reference's counter quirk included)
//   xm    : uint32[]        1 bit per 1024-base block: block holds a non-ACGT base or a base whose
//                           deletion bias hp_del_bias[hp] differs from 1 ("exceptional" block)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pb {

constexpr int kXmShift = 10;  // exception bitmap granularity: 1024 bases

__device__ __forceinline__ uint32_t base_code(uint8_t c, bool &ok) {
  // A=0 C=1 G=2 T=3
  switch (c) {
    case 'A': ok = true; return 0u;
    case 'C': ok = true; return 1u;
    case 'G': ok = true; return 2u;
    case 'T': ok = true; return 3u;
    default: ok = false; return 0u;
  }
}

// synthetic i.i.d. ACGT text (benchmarks): one 64-bit hash per 16 bases
__global__ void k_synth_ascii(uint8_t *ascii, int64_t len, uint64_t seed) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i0 = w * 16;
  if (i0 >= len) return;
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(w + 1);  // splitmix64
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  const uint32_t lut = 0x54474341u;  // "ACGT"
  uint32_t out[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint32_t v = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const uint32_t code = (uint32_t)(z >> (2 * (q * 4 + b))) & 3u;
      v |= ((lut >> (8 * code)) & 0xFFu) << (8 * b);
    }
    out[q] = v;
  }
  if (i0 + 16 <= len) {
    *reinterpret_cast<uint4 *>(ascii + i0) = make_uint4(out[0], out[1], out[2], out[3]);
  } else {
    for (int64_t i = i0; i < len; ++i) ascii[i] = (uint8_t)(out[(i - i0) >> 2] >> (8 * ((i - i0) & 3)));
  }
}

// upper-case in place (toupper in the C locale, :1035-1037), pack, flag non-ACGT blocks.
// One thread per 16 bases; `ascii` is padded to a multiple of 16 with zeros.
__global__ void k_upper_pack(uint8_t *ascii, int64_t len, uint32_t *pk, uint32_t *xm) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i0 = w * 16;
  if (i0 >= len) return;
  uint4 v = *reinterpret_cast<const uint4 *>(ascii + i0);
  uint32_t in[4] = {v.x, v.y, v.z, v.w};
  uint32_t word = 0;
  bool any_bad = false;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint32_t o = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      uint8_t c = (uint8_t)(in[q] >> (8 * b));
      if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32);
      o |= (uint32_t)c << (8 * b);
      bool ok;
      const uint32_t code = base_code(c, ok);
      if (i0 + q * 4 + b < len) {
        word |= code << (2 * (q * 4 + b));
        any_bad |= !ok;
      }
    }
    in[q] = o;
  }
  *reinterpret_cast<uint4 *>(ascii + i0) = make_uint4(in[0], in[1], in[2], in[3]);
  pk[w] = word;
  if (any_bad) {
    const int64_t blk = i0 >> kXmShift;
    atomicOr(&xm[blk >> 5], 1u << (blk & 31));
  }
}

// hp[] with the reference's counter: run length L -> L (L <= 11), else 11 / 10 alternating
// (nnum > 11 -> 10, :1046-1048); every base of an 'N' run gets 1 (:1050-1054).
// One thread per 2 bases (one hp4 byte).  Walks are capped; a capped walk raises *flag so the
// engine can fall back to a host scan for pathological inputs (megabase homopolymers).
__device__ __forceinline__ uint32_t hp_of(const uint8_t *ascii, int64_t len, int64_t i, uint32_t *flag) {
  const uint8_t c = ascii[i];
  if (c == 'N') return 1u;
  const int64_t cap = 1 << 16;
  int64_t l = 0, r = 0;
  while (i - l - 1 >= 0 && ascii[i - l - 1] == c && l < cap) ++l;
  while (i + r + 1 < len && ascii[i + r + 1] == c && r < cap) ++r;
  if (l >= cap || r >= cap) *flag = 1u;
  const int64_t L = l + r + 1;
  if (L <= 11) return (uint32_t)L;
  return ((L - 11) & 1) ? 10u : 11u;
}

// One thread per 8 bases (one 32-bit word of hp4), CTAs stride over the sequence.  Runs inside the thread's 8 bytes are
// measured in registers; only a run that touches the group's first or last byte is followed into the neighbouring
// text, and only when that byte is not 'N' (N runs of any length are accepted).  A walk capped at 65 536 bases raises
// *flag: the engine refuses a homopolymer of another letter that long.  The histogram is summed per warp (packed
// 16-bit counters, REDUX) before it touches shared memory, and every CTA adds its 12 cells to the global histogram
// once: the one-thread-per-2-bases version spent its time in same-address atomics (1.3 ms per 242 Mbp; this one is
// bound by the text it reads).
constexpr int kHpThreads = 256;
__global__ void __launch_bounds__(kHpThreads) k_hp(const uint8_t *__restrict__ ascii, int64_t len, uint8_t *hp4,
                                                   uint32_t *xm, unsigned long long *hpfreq,
                                                   const uint8_t *bias_is_one /*[12]*/, uint32_t *flag) {
  __shared__ unsigned int hist[12];
  __shared__ unsigned int not_one;  // bit h: hp_del_bias[h] != 1
  if (threadIdx.x < 12) hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    unsigned int m = 0;
    for (int h = 0; h < 12; ++h) m |= bias_is_one[h] ? 0u : 1u << h;
    not_one = m;
  }
  __syncthreads();
  const uint32_t special_mask = not_one;
  const uint32_t lane = threadIdx.x & 31u;
  const int64_t n_groups = (len + 7) / 8;
  const int64_t n_iter = (n_groups + (int64_t)gridDim.x * kHpThreads - 1) / ((int64_t)gridDim.x * kHpThreads);
  for (int64_t it = 0; it < n_iter; ++it) {
    const int64_t t = (it * gridDim.x + blockIdx.x) * kHpThreads + threadIdx.x;
    const int64_t i0 = t * 8;
    unsigned long long cnt4 = 0;  // 12 bins x 4 bits (a thread counts at most 8 bases)
    if (i0 < len) {
      // the text is zero-padded to a multiple of 16 (+64) behind len: bytes past the end compare unequal to any base
      const uint2 v = *reinterpret_cast<const uint2 *>(ascii + i0);
      uint8_t b[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = (uint8_t)((j < 4 ? v.x : v.y) >> (8 * (j & 3)));
      const int64_t cap = 1 << 16;
      int64_t l = 0, r = 0;
      // left[0] / right[7] only reach bytes equal to b[0] / b[7]; an 'N' gets hp 1 whatever its run: no walk
      if (b[0] != 'N')
        while (i0 - l - 1 >= 0 && ascii[i0 - l - 1] == b[0] && l < cap) ++l;
      if (b[7] != 'N')
        while (i0 + 7 + r + 1 < len && ascii[i0 + 7 + r + 1] == b[7] && r < cap) ++r;
      if (l >= cap || r >= cap) *flag = 1u;
      uint32_t left[8], right[8];
      left[0] = (uint32_t)l;
#pragma unroll
      for (int j = 1; j < 8; ++j) left[j] = b[j] == b[j - 1] ? left[j - 1] + 1u : 0u;
      right[7] = (uint32_t)r;
#pragma unroll
      for (int j = 6; j >= 0; --j) right[j] = b[j] == b[j + 1] ? right[j + 1] + 1u : 0u;
      uint32_t word = 0;
      bool special = false;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (i0 + j < len) {
          const uint32_t L = left[j] + right[j] + 1u;
          const uint32_t h = b[j] == 'N' ? 1u : (L <= 11u ? L : (((L - 11u) & 1u) ? 10u : 11u));
          word |= h << (4 * j);
          cnt4 += 1ull << (4u * h);
          special |= ((special_mask >> h) & 1u) != 0u;
        }
      }
      *reinterpret_cast<uint32_t *>(hp4 + t * 4) = word;
      if (special) {
        const int64_t blk = i0 >> kXmShift;
        atomicOr(&xm[blk >> 5], 1u << (blk & 31));
      }
    }
    // two bins per word in 16-bit fields for the warp sums (at most 256 bases per warp: no overflow)
    uint32_t mine = 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const uint32_t two = (uint32_t)(cnt4 >> (8 * k));
      const uint32_t s = __reduce_add_sync(0xFFFFFFFFu, (two & 0xFu) | ((two & 0xF0u) << 12));
      if ((lane >> 1) == (uint32_t)k) mine = (lane & 1u) ? (s >> 16) : (s & 0xFFFFu);
    }
    if (lane < 12u && mine) atomicAdd(&hist[lane], mine);
  }
  __syncthreads();
  if (threadIdx.x < 12 && hist[threadIdx.x]) atomicAdd(&hpfreq[threadIdx.x], (unsigned long long)hist[threadIdx.x]);
}

// ---- sequence sets (--strategy trans / templ): many short sequences concatenated into one device text ----------
// start[n+1]: first base of every sequence in the concatenation.  Homopolymer runs end at sequence boundaries and
// windows never cross them, so everything downstream of K0 treats the concatenation like one genome.

// index of the sequence holding base i (largest t with start[t] <= i)
__device__ __forceinline__ uint32_t set_find(const uint32_t *__restrict__ start, uint32_t n, uint32_t i) {
  uint32_t lo = 0, hi = n;  // start[lo] <= i < start[hi]
  while (hi - lo > 1u) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(&start[mid]) <= i) lo = mid;
    else hi = mid;
  }
  return lo;
}

// The reference upper-cases these sequences with `for (i = 1; i <= len; i++)` everywhere except in
// simulate_by_qshmm_trans (pbsim.cpp:3330, :4474, :5049 vs :2774): the first base keeps its case.
__global__ void k_set_save_first(const uint8_t *ascii, const uint32_t *start, uint32_t n, uint8_t *first) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) first[t] = ascii[start[t]];
}
__global__ void k_set_restore_first(uint8_t *ascii, const uint32_t *start, uint32_t n, const uint8_t *first,
                                    uint32_t *pk, uint32_t *xm) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint8_t c = first[t];
  if (c < 'a' || c > 'z') return;
  const uint32_t i = start[t];
  if (start[t + 1] == i) return;  // empty sequence
  ascii[i] = c;                   // a lower-case letter is not one of A, C, G, T: the base is exceptional
  atomicAnd(&pk[i >> 4], ~(3u << (2u * (i & 15u))));
  const uint32_t blk = i >> kXmShift;
  atomicOr(&xm[blk >> 5], 1u << (blk & 31));
}

__device__ __forceinline__ uint32_t hp_of_bounded(const uint8_t *ascii, int64_t lo, int64_t hi, int64_t i,
                                                  uint32_t *flag) {
  const uint8_t c = ascii[i];
  if (c == 'N') return 1u;
  const int64_t cap = 1 << 16;
  int64_t l = 0, r = 0;
  while (i - l - 1 >= lo && ascii[i - l - 1] == c && l < cap) ++l;
  while (i + r + 1 < hi && ascii[i + r + 1] == c && r < cap) ++r;
  if (l >= cap || r >= cap) *flag = 1u;
  const int64_t L = l + r + 1;
  if (L <= 11) return (uint32_t)L;
  return ((L - 11) & 1) ? 10u : 11u;
}

// k_hp for a sequence set; hpfreq counts every base weight[t] times (transcripts: plus + minus reads, the
// --hp-del-bias prepass of pbsim.cpp:2714-2718; templates: weight == nullptr, 1)
__global__ void k_hp_set(const uint8_t *ascii, int64_t len, const uint32_t *start, uint32_t n, const uint32_t *weight,
                         uint8_t *hp4, uint32_t *xm, unsigned long long *hpfreq, const uint8_t *bias_is_one,
                         uint32_t *flag) {
  __shared__ unsigned long long hist[12];
  if (threadIdx.x < 12) hist[threadIdx.x] = 0;
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i0 = t * 2;
  if (i0 < len) {
    uint32_t q = set_find(start, n, (uint32_t)i0);
    uint32_t h[2] = {0, 0};
    bool special = false;
    for (int k = 0; k < 2; ++k) {
      const int64_t i = i0 + k;
      if (i >= len) break;
      while (i >= (int64_t)start[q + 1]) ++q;  // skips empty sequences too
      h[k] = hp_of_bounded(ascii, start[q], start[q + 1], i, flag);
      atomicAdd(&hist[h[k]], (unsigned long long)(weight ? weight[q] : 1u));
      special |= !bias_is_one[h[k]];
    }
    hp4[t] = (uint8_t)(h[0] | (h[1] << 4));
    if (special) {
      const int64_t blk = i0 >> kXmShift;
      atomicOr(&xm[blk >> 5], 1u << (blk & 31));
    }
  }
  __syncthreads();
  if (threadIdx.x < 12 && hist[threadIdx.x]) atomicAdd(&hpfreq[threadIdx.x], hist[threadIdx.x]);
}

// true if any 1024-base block overlapping genome range [g0, g1] is exceptional
__device__ __forceinline__ bool range_exceptional(const uint32_t *__restrict__ xm, uint32_t g0, uint32_t g1) {
  const uint32_t b0 = g0 >> kXmShift, b1 = g1 >> kXmShift;
  for (uint32_t w = b0 >> 5; w <= (b1 >> 5); ++w) {
    uint32_t bits = __ldg(&xm[w]);
    if (w == (b0 >> 5)) bits &= 0xFFFFFFFFu << (b0 & 31);
    if (w == (b1 >> 5)) bits &= 0xFFFFFFFFu >> (31 - (b1 & 31));
    if (bits) return true;
  }
  return false;
}

}  // namespace pb
