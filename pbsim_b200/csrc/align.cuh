// K5 — option "align": each (read, pass)'s true alignment as one SAM line instead of its MAF block.
//
// Pass 2 renders the MAF block of every record as usual, into a scratch stream; these kernels turn each block into a
// SAM alignment line (DESIGN §2.10).  The MAF kernels therefore run unchanged: the alignment columns are taken from the
// one place that already renders them, both rows in reference order (minus-strand rows are mirrored there).
//
// Column classes, from the two MAF bytes of a column: '-' in the reference row is an insertion, '-' in the read row a
// deletion, equal bytes a match ('='), different bytes a substitution ('X').  That equals the event kind: a
// substitution draws from an alphabet without the window base (set_mut, pbsim.cpp:5481-5486; :2235-2246), and where
// the reference base is not one of A/C/G/T the read base is one (the "ATGC" alphabet) and the reference byte is not; on
// the minus strand both bytes are complemented by the same map (comp_char), which is one-to-one.
//
// One warp per record.  k_aln_sizes finds the first and last '='/'X' column, counts the insertions (soft clip) and
// deletions (dropped, POS moves past them) outside them, and walks the runs between them to size the CIGAR; k_aln_write
// walks the same runs again and writes them, the closing lane of each run at an offset from a warp scan.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "emit.cuh"

namespace pb {

constexpr uint32_t kAlnMatch = 0u, kAlnSub = 1u, kAlnIns = 2u, kAlnDel = 3u, kAlnNone = 4u;

__host__ __device__ __forceinline__ uint32_t aln_op(uint8_t ref, uint8_t read) {
  if (ref == '-') return kAlnIns;
  if (read == '-') return kAlnDel;
  return ref == read ? kAlnMatch : kAlnSub;
}

// what k_aln_sizes leaves for k_aln_write, per sub-read
struct AlnRec {
  uint32_t c_lo, c_hi;        // columns [c_lo, c_hi) between the first and the last '='/'X' column (c_lo = c_hi: unmapped)
  uint32_t clip_lo, clip_hi;  // insertions in front of c_lo / behind c_hi: the soft clips
  uint32_t pos;               // 1-based POS (0: unmapped)
  uint32_t nm;                // X + I + D columns in [c_lo, c_hi)
  uint32_t cigar_len;         // characters of the CIGAR, clips included
  uint32_t core_len;          // characters of the runs in [c_lo, c_hi)
};

struct AlnArgs {
  DeviceSet S;
  Batch B;
  EmitParams P;
  uint32_t n_sub;
  const EmitLay *lay;
  const uint64_t *reads_off, *maf_off;
  const uint8_t *reads, *maf;  // the sub-reads' reads records and MAF blocks
  const uint8_t *rname;        // WGS: the sequence's name (RNAME)
  uint32_t rname_len;
  AlnRec *rec;
  const uint64_t *sam_off;
  uint8_t *sam;
};

__device__ __forceinline__ uint32_t aln_qname_len(const EmitParams &P, uint64_t read_id, uint32_t pass) {
  return P.id_head_len + 1u + ndigits(read_id) + (P.sam ? 1u + ndigits(pass) : 0u);
}

// The runs of columns [c0, c1): calls put(op, len, at) once per run, on the lane that closes it, where `at` counts the
// characters ("<len><op>") of the runs in front of it.  Returns the characters of all runs; *nm: the X / I / D columns.
template <class Put>
__device__ __forceinline__ uint32_t aln_runs(const uint8_t *__restrict__ ref, const uint8_t *__restrict__ rd, uint32_t c0,
                                             uint32_t c1, uint32_t lane, uint32_t *nm, Put put) {
  uint32_t chars = 0, nmt = 0, open_op = kAlnNone, open_start = c0;
  for (uint32_t base = c0; base < c1; base += 32u) {
    const uint32_t c = base + lane;
    const bool valid = c < c1;
    const uint32_t op = valid ? aln_op(__ldg(ref + c), __ldg(rd + c)) : kAlnNone;
    uint32_t prev = __shfl_up_sync(0xFFFFFFFFu, op, 1);
    if (lane == 0) prev = open_op;
    const bool start = valid && op != prev;
    const uint32_t m_start = __ballot_sync(0xFFFFFFFFu, start);
    // a run that starts at c > c0 closes the run in front of it, which began at the previous start
    const uint32_t below = m_start & ((1u << lane) - 1u);
    const uint32_t pstart = below ? base + 31u - __clz(below) : open_start;
    const bool close = start && c != c0;
    const uint32_t len = c - pstart;
    const uint32_t w = close ? ndigits(len) + 1u : 0u;
    uint32_t x = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (uint32_t)o) x += y;
    }
    if (close) put(prev, len, chars + x - w);
    chars += __shfl_sync(0xFFFFFFFFu, x, 31);
    nmt += __reduce_add_sync(0xFFFFFFFFu, (close && prev != kAlnMatch) ? len : 0u);
    if (m_start) open_start = base + 31u - __clz(m_start);
    const uint32_t last = min(31u, c1 - 1u - base);
    open_op = __shfl_sync(0xFFFFFFFFu, op, last);
  }
  if (c1 > c0) {  // the last run ends at c1
    const uint32_t len = c1 - open_start;
    if (lane == 0) put(open_op, len, chars);
    chars += ndigits(len) + 1u;
    if (open_op != kAlnMatch) nmt += len;
  }
  *nm = nmt;
  return chars;
}

// the fixed-width fields of a record: RNAME of its sequence
__device__ __forceinline__ void aln_rname(const AlnArgs &A, const RefName &N, const uint8_t **p, uint32_t *n) {
  if (N.ptr) { *p = N.ptr; *n = N.len; }
  else { *p = A.rname; *n = A.rname_len; }
}

__global__ void __launch_bounds__(256) k_aln_sizes(const __grid_constant__ AlnArgs A, uint64_t *sam_size) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp0 = blockIdx.x * (blockDim.x / 32u) + (threadIdx.x >> 5);
  const uint32_t nwarps = gridDim.x * (blockDim.x / 32u);
  for (uint32_t s = warp0; s < A.n_sub; s += nwarps) {
    const uint32_t r = s / A.P.pass_num, pass = s % A.P.pass_num;
    const uint32_t ncol = A.B.ncol[s], rlen = A.B.rlen[s];
    const EmitLay L = A.lay[s];
    const uint8_t *mf = A.maf + A.maf_off[s];
    const uint8_t *ref = mf + L.refrow_rel, *rd = mf + L.readrow_rel;
    // first / last '='/'X' column, the insertions and deletions outside them, all insertions
    uint32_t c_lo = 0xFFFFFFFFu, c_hi = 0, lead_i = 0, lead_d = 0, trail_i = 0, ins = 0;
    for (uint32_t base = 0; base < ncol; base += 32u) {
      const uint32_t c = base + lane;
      const uint32_t op = c < ncol ? aln_op(__ldg(ref + c), __ldg(rd + c)) : kAlnNone;
      const uint32_t m_mx = __ballot_sync(0xFFFFFFFFu, op <= kAlnSub);
      const uint32_t m_i = __ballot_sync(0xFFFFFFFFu, op == kAlnIns);
      const uint32_t m_d = __ballot_sync(0xFFFFFFFFu, op == kAlnDel);
      ins += __popc(m_i);
      if (c_lo == 0xFFFFFFFFu) {
        const uint32_t front = m_mx ? (1u << (__ffs(m_mx) - 1u)) - 1u : 0xFFFFFFFFu;  // lanes in front of the first
        lead_i += __popc(m_i & front);
        lead_d += __popc(m_d & front);
        if (m_mx) c_lo = base + __ffs(m_mx) - 1u;
      }
      if (m_mx) {
        const uint32_t hi = 31u - __clz(m_mx);
        c_hi = base + hi + 1u;
        trail_i = __popc(m_i >> hi);  // bit hi is not an insertion
      } else {
        trail_i += __popc(m_i);
      }
    }
    const RefName N = ref_name(A.S, A.B, r, A.P.glen);
    const uint32_t minus = (A.B.plan_meta[r] >> 8) & 1u;
    AlnRec R;
    R.nm = 0;
    R.core_len = 0;
    if (c_lo == 0xFFFFFFFFu) {  // no '=' / 'X' column: unmapped
      R.c_lo = R.c_hi = 0;
      R.clip_lo = R.clip_hi = 0;
      R.pos = 0;
      R.cigar_len = 1u;
    } else {
      R.c_lo = c_lo;
      R.c_hi = c_hi;
      R.clip_lo = lead_i;
      R.clip_hi = trail_i;
      // the MAF block's reference row starts at the window's first base on the plus strand; a minus-strand read that
      // ended before its window was used up (--method sample, :1775-1833) starts that many bases further right
      const uint32_t consumed = ncol - ins;
      const uint32_t wlen = A.B.plan_wlen[r];
      R.pos = N.off + (minus && wlen > consumed ? wlen - consumed : 0u) + lead_d + 1u;
      uint32_t nm = 0;
      R.core_len = aln_runs(ref, rd, c_lo, c_hi, lane, &nm, [](uint32_t, uint32_t, uint32_t) {});
      R.nm = nm;
      R.cigar_len = R.core_len + (lead_i ? ndigits(lead_i) + 1u : 0u) + (trail_i ? ndigits(trail_i) + 1u : 0u);
    }
    if (lane == 0) {
      const uint64_t read_id = A.B.first_read + 1u + r;
      const uint8_t *rn;
      uint32_t rn_len;
      aln_rname(A, N, &rn, &rn_len);
      const bool mapped = R.pos != 0u;
      const uint32_t flag = mapped ? (minus ? 16u : 0u) : 4u;
      const uint32_t seq = rlen ? rlen : 1u;
      uint64_t n = aln_qname_len(A.P, read_id, pass) + 1u + ndigits(flag) + 1u + (mapped ? rn_len : 1u) + 1u +
                   ndigits(R.pos) + 1u + (mapped ? 2u : 1u) + 1u + R.cigar_len;
      n += PB_LEN("\t*\t0\t0\t") + seq + 1u + seq + PB_LEN("\tNM:i:") + ndigits(R.nm) + 1u;
      sam_size[s] = n;
      A.rec[s] = R;
    }
  }
}

__global__ void __launch_bounds__(256) k_aln_write(const __grid_constant__ AlnArgs A) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp0 = blockIdx.x * (blockDim.x / 32u) + (threadIdx.x >> 5);
  const uint32_t nwarps = gridDim.x * (blockDim.x / 32u);
  for (uint32_t s = warp0; s < A.n_sub; s += nwarps) {
    const uint32_t r = s / A.P.pass_num, pass = s % A.P.pass_num;
    const uint32_t rlen = A.B.rlen[s];
    const uint32_t minus = (A.B.plan_meta[r] >> 8) & 1u;
    const EmitLay L = A.lay[s];
    const AlnRec R = A.rec[s];
    const uint64_t read_id = A.B.first_read + 1u + r;
    const bool mapped = R.pos != 0u;
    uint8_t *o = A.sam + A.sam_off[s];
    // QNAME .. MAPQ and the front clip
    const uint32_t qn = aln_qname_len(A.P, read_id, pass);
    const uint32_t flag = mapped ? (minus ? 16u : 0u) : 4u;
    const RefName N = ref_name(A.S, A.B, r, A.P.glen);
    const uint8_t *rn;
    uint32_t rn_len;
    aln_rname(A, N, &rn, &rn_len);
    const uint32_t head = qn + 1u + ndigits(flag) + 1u + (mapped ? rn_len : 1u) + 1u + ndigits(R.pos) + 1u +
                          (mapped ? 2u : 1u) + 1u;
    uint8_t *cig = o + head;
    const uint32_t front = R.clip_lo ? ndigits(R.clip_lo) + 1u : 0u;
    if (lane == 0) {
      RecLayout RL;
      RL.d_rid = ndigits(read_id);
      RL.d_pass = ndigits(pass);
      uint8_t *p = put_id(o, A.P, read_id, pass, RL);
      *p++ = '\t';
      p = put_dec(p, flag, ndigits(flag));
      *p++ = '\t';
      if (mapped) p = put_mem(p, reinterpret_cast<const char *>(rn), rn_len);
      else *p++ = '*';
      *p++ = '\t';
      p = put_dec(p, R.pos, ndigits(R.pos));
      *p++ = '\t';
      if (mapped) { *p++ = '6'; *p++ = '0'; }
      else *p++ = '0';
      *p++ = '\t';
      if (!mapped) {
        *p++ = '*';
      } else {
        if (R.clip_lo) { p = put_dec(p, R.clip_lo, ndigits(R.clip_lo)); *p++ = 'S'; }
        p = cig + front + R.core_len;
        if (R.clip_hi) { p = put_dec(p, R.clip_hi, ndigits(R.clip_hi)); *p++ = 'S'; }
      }
    }
    // the runs
    if (mapped) {
      const uint8_t *mf = A.maf + A.maf_off[s];
      uint8_t *core = cig + front;
      uint32_t nm;
      aln_runs(mf + L.refrow_rel, mf + L.readrow_rel, R.c_lo, R.c_hi, lane, &nm,
               [&](uint32_t op, uint32_t len, uint32_t at) {
                 uint8_t *q = put_dec(core + at, len, ndigits(len));
                 *q = (uint8_t)(0x4449583Du >> (8u * op));  // "=XID"
               });
    }
    // RNEXT PNEXT TLEN, SEQ and QUAL in reference orientation, the tag
    uint8_t *p = cig + R.cigar_len;
    const uint32_t seq = rlen ? rlen : 1u;
    if (lane == 0) {
      PB_PUT_LIT(p, "\t*\t0\t0\t");
      p[PB_LEN("\t*\t0\t0\t") + seq] = '\t';
      uint8_t *t = p + PB_LEN("\t*\t0\t0\t") + 2u * seq + 1u;
      t = PB_PUT_LIT(t, "\tNM:i:");
      t = put_dec(t, R.nm, ndigits(R.nm));
      *t = '\n';
      if (rlen == 0) {
        p[PB_LEN("\t*\t0\t0\t")] = '*';
        p[PB_LEN("\t*\t0\t0\t") + 2u] = '*';
      }
    }
    uint8_t *sq = p + PB_LEN("\t*\t0\t0\t"), *ql = sq + seq + 1u;
    const uint8_t *rs = A.reads + A.reads_off[s] + L.seq_rel, *rq = A.reads + A.reads_off[s] + L.qual_rel;
    for (uint32_t j = lane; j < rlen; j += 32u) {
      const uint32_t src = minus ? rlen - 1u - j : j;
      const uint8_t b = __ldg(rs + src);
      sq[j] = minus ? comp_char(b) : b;
      ql[j] = __ldg(rq + src);
    }
  }
}

}  // namespace pb
