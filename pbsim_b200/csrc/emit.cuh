// K4 — pass 2: event streams -> FASTQ / SAM / MAF bytes, written in read order.
// Replaces the reference's record emission (pbsim.cpp:2318-2383 = :4012-4078), count_digit (:5823)
// and the three revcomp calls per minus-strand read (:5841): minus-strand reads are generated on the
// reverse-complemented window and their MAF rows are mirrored back while being written.
//
// Work unit: one warp formats one tile of PB_TILE events of one (read, pass).  Tiles are independent
// thanks to the checkpoints pass 1 left; output positions come from warp ballots / a warp prefix
// scan over deletion counts, so every store lands at its final byte and consecutive lanes write
// consecutive bytes.  The genome is read from the 2-bit packed array (coalesced; neighbouring lanes
// share words); tiles that touch an exceptional 1024-base block read the ASCII copy instead.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "k0_genome.cuh"
#include "sim_kernels.cuh"

namespace pb {

constexpr int kEmitThreads = 256;
constexpr int kEmitWarps = kEmitThreads / 32;

struct EmitParams {
  uint32_t pass_num;
  uint32_t sam;            // 0: FASTQ, 1: SAM records (pass_num > 1), 2: BAM records (same content, binary)
  uint32_t id_head_len;    // strlen(id_prefix + seq_num)
  char id_head[160];       // "<id_prefix><seq_num>"
  uint32_t rq_len;
  char rq[32];             // printf("%f", accuracy_mean)
  float rq_f;              // the same text read back as a float (BAM: rq:f)
  uint32_t glen;
  uint32_t qs_segments;    // method is qshmm: segmented sub-reads use one slot per tile
  uint32_t sample;         // --method sample: the MAF line reports the bases consumed, not the window (:1847)
};

// the reference-row naming of a record: WGS writes "ref" and the sequence length; the transcript / template
// strategies the sequence's own name, positions relative to it and its length (pbsim.cpp:2968-2996, :3486-3514)
struct RefName {
  const uint8_t *ptr;   // nullptr: "ref"
  uint32_t len;         // characters written
  uint32_t width;       // digit_num1[0]: strlen(id) for transcripts, 3 for WGS and (sic) templates
  uint32_t src_len;     // genome.len / transcript.len / templ.len
  uint32_t off;         // mut.seq_left - 1
};

__device__ __forceinline__ RefName ref_name(const DeviceSet &S, const Batch &B, uint32_t r, uint32_t glen) {
  RefName N;
  if (S.strategy == PBSIM_STRATEGY_WGS) {
    N.ptr = nullptr;
    N.len = 3u;
    N.width = 3u;
    N.src_len = glen;
    N.off = B.plan_off[r];
    return N;
  }
  const uint32_t t = B.plan_tr[r];
  N.ptr = S.ids + S.id_start[t];
  N.len = S.id_start[t + 1] - S.id_start[t];
  N.width = S.strategy == PBSIM_STRATEGY_TRANS ? N.len : 3u;
  N.src_len = S.start[t + 1] - S.start[t];
  N.off = B.plan_off[r] - S.start[t];
  return N;
}

// where the per-base rows of a sub-read's records start (relative to the record); computed once per sub-read by
// k_sizes so that the tiles of pass 2 load it instead of re-deriving digit counts
struct EmitLay {
  uint32_t seq_rel, qual_rel, ip_rel, pw_rel, refrow_rel, readrow_rel;
};

struct EmitArgs {
  DeviceSet S;
  PhiloxKeys keys;             // PHILOX mode: pass 2 re-derives the 4-way choice of substitutions on non-ACGT bases
  uint32_t philox;
  DeviceGenome G;
  Batch B;
  EmitParams P;
  const uint8_t *ev;
  const Ckpt *ck;
  uint32_t n_sub;              // valid subreads (after the quota cut)
  uint64_t n_tiles;
  const uint64_t *tile_start;  // [n_sub + 1]
  const uint32_t *tile_sub;    // [n_tiles] sub-read of a tile (k_tile_desc)
  struct TileDesc *desc;       // [n_tiles] everything pass 2 needs to know about a tile (k_tile_desc)
  const EmitLay *lay;          // [n_sub] row positions inside the records (k_sizes)
  const uint64_t *reads_off;   // [n_sub + 1]
  const uint64_t *maf_off;     // [n_sub + 1]
  uint8_t *out_reads;
  uint8_t *out_maf;
};

__host__ __device__ __forceinline__ uint32_t ndigits(uint64_t v) {  // count_digit (:5823), without divisions
  if (v < 100000ull) return v < 10ull ? 1u : (v < 100ull ? 2u : (v < 1000ull ? 3u : (v < 10000ull ? 4u : 5u)));
  if (v < 10000000000ull)
    return v < 1000000ull ? 6u : (v < 10000000ull ? 7u : (v < 100000000ull ? 8u : (v < 1000000000ull ? 9u : 10u)));
  uint32_t d = 10;
  for (v /= 10000000000ull; v; v /= 10) ++d;
  return d;
}

struct RecLayout {
  uint32_t idlen, d_rid, d_pass;
  uint64_t seq_rel, qual_rel, ip_rel, pw_rel, tail_rel, reads_size;
  uint32_t pa[4], pb_[4];  // MAF padding of the ref row / the read row fields
  uint32_t d_off, d_wlen, d_glen, d_rlen;
  uint64_t refrow_rel, readrow_rel, maf_size;
};

#define PB_SAM_S1 "\t4\t*\t0\t255\t*\t*\t0\t0\t"
#define PB_SAM_S2 "\tcx:i:3\tip:B:C"
#define PB_SAM_S3 "\tnp:i:1\tpw:B:C"
#define PB_SAM_S4 "\tqs:i:0\tqe:i:"
#define PB_SAM_S5 "\trq:f:"
#define PB_SAM_S6 "\tsn:B:f,10.0,10.0,10.0,10.0\tzm:i:"
#define PB_SAM_S7 "\tRG:Z:ffffffff\n"
#define PB_LEN(s) ((uint32_t)(sizeof(s) - 1))

// integer tags take the smallest type that holds the value, as htslib's SAM parser chooses it
__device__ __forceinline__ uint32_t bam_int_width(int64_t v) {
  if (v < 0) return v >= -128 ? 1u : (v >= -32768 ? 2u : 4u);
  return v <= 255 ? 1u : (v <= 65535 ? 2u : 4u);
}
__device__ __forceinline__ uint8_t bam_int_type(int64_t v) {
  if (v < 0) return v >= -128 ? 'c' : (v >= -32768 ? 's' : 'i');
  return v <= 255 ? 'C' : (v <= 65535 ? 'S' : 'I');
}
// 4-bit base codes "=ACMGRSVTWYHKDBN" (SAM spec 4.2.3); anything else is N, lower case counts as upper case
__device__ __forceinline__ uint32_t bam_nibble(uint8_t c) {
  if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32);
  switch (c) {
    case '=': return 0u;  case 'A': return 1u;  case 'C': return 2u;  case 'M': return 3u;
    case 'G': return 4u;  case 'R': return 5u;  case 'S': return 6u;  case 'V': return 7u;
    case 'T': return 8u;  case 'W': return 9u;  case 'Y': return 10u; case 'H': return 11u;
    case 'K': return 12u; case 'D': return 13u; case 'B': return 14u; default: return 15u;
  }
}
// BAM base bytes that two writers share (two bases per byte): OR the bits into the zeroed record
__device__ __forceinline__ void atomic_or_byte(uint8_t *b, uint32_t bits) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(b);
  atomicOr(reinterpret_cast<unsigned int *>(a & ~(uintptr_t)3), bits << (8u * (uint32_t)(a & 3u)));
}
// one read base into its row(s): text formats store characters; BAM packs two bases per byte (high nibble first)
// with an atomic OR into the zeroed record, and stores the quality value itself
template <bool BAM>
__device__ __forceinline__ void put_read_base(uint8_t *seq, uint8_t *qual, uint32_t Pp, uint8_t ch, uint32_t nib,
                                              uint32_t qv, bool has_qv) {
  if (!BAM) {
    seq[Pp] = ch;
    qual[Pp] = has_qv ? (uint8_t)(qv + 33u) : (uint8_t)'!';
  } else {
    atomic_or_byte(seq + (Pp >> 1), nib << ((Pp & 1u) ? 0u : 4u));
    qual[Pp] = has_qv ? (uint8_t)qv : (uint8_t)0;
  }
}

__device__ __forceinline__ RecLayout rec_layout(const EmitParams &P, const RefName &N, uint64_t read_id, uint32_t pass,
                                                uint32_t wlen, uint32_t rlen, uint32_t ncol) {
  const uint32_t offset = N.off;
  RecLayout L;
  L.d_rid = ndigits(read_id);
  L.d_pass = ndigits(pass);
  const uint32_t qe_digits = rlen == 0 ? 2u : ndigits(rlen - 1u);  // "-1" when the read is empty
  if (!P.sam) {
    L.idlen = P.id_head_len + 1u + L.d_rid;  // "<head>_<read>"
    L.seq_rel = 1u + L.idlen + 1u;
    L.qual_rel = L.seq_rel + rlen + 2u + L.idlen + 1u;
    L.reads_size = L.qual_rel + rlen + 1u;
    L.ip_rel = L.pw_rel = L.tail_rel = 0;
  } else if (P.sam == 2u) {
    // BAM alignment record (SAM spec 4.2) of an unmapped read: 36 fixed bytes, name + NUL, 4-bit bases, qualities,
    // then the tags with the types samtools gives them when it converts the reference's SAM text
    L.idlen = P.id_head_len + 1u + L.d_rid + 1u + L.d_pass;
    L.seq_rel = 36u + L.idlen + 1u;
    L.qual_rel = L.seq_rel + (rlen + 1u) / 2u;
    L.ip_rel = L.qual_rel + rlen + 4u + 8u;          // cx:C (4), ip:B:C header (8)
    L.pw_rel = L.ip_rel + rlen + 4u + 8u;            // np:C (4), pw:B:C header (8)
    L.tail_rel = L.pw_rel + rlen;
    const int64_t qe = (int64_t)rlen - 1;
    L.reads_size = L.tail_rel + 4u + (3u + bam_int_width(qe)) + 7u + 24u + (3u + bam_int_width((int64_t)read_id)) + 12u;
  } else {
    L.idlen = P.id_head_len + 1u + L.d_rid + 1u + L.d_pass;  // "<head>/<read>/<pass>"
    L.seq_rel = L.idlen + PB_LEN(PB_SAM_S1);
    L.qual_rel = L.seq_rel + rlen + 1u;
    L.ip_rel = L.qual_rel + rlen + PB_LEN(PB_SAM_S2);
    L.pw_rel = L.ip_rel + 2ull * rlen + PB_LEN(PB_SAM_S3);
    L.tail_rel = L.pw_rel + 2ull * rlen;
    L.reads_size = L.tail_rel + PB_LEN(PB_SAM_S4) + qe_digits + PB_LEN(PB_SAM_S5) + P.rq_len + PB_LEN(PB_SAM_S6) +
                   L.d_rid + PB_LEN(PB_SAM_S7);
  }
  // MAF field widths (:2336-2350); note the name column assumes an id of 1 + digits(read number)
  L.d_off = ndigits(offset);
  L.d_wlen = ndigits(wlen);
  L.d_glen = ndigits(N.src_len);
  L.d_rlen = ndigits(rlen);
  const uint32_t d1[4] = {N.width, L.d_off, L.d_wlen, L.d_glen};
  const uint32_t d2[4] = {1u + L.d_rid, 1u, L.d_rlen, L.d_rlen};
  for (int i = 0; i < 4; ++i) {
    const uint32_t dn = d1[i] > d2[i] ? d1[i] : d2[i];
    L.pa[i] = dn - d1[i];
    L.pb_[i] = dn - d2[i];
  }
  // "a\ns " name pa0 pa1 " off" pa2 " wlen +" pa3 " glen " ROW "\n"
  L.refrow_rel = 4u + N.len + L.pa[0] + L.pa[1] + 1u + L.d_off + L.pa[2] + 1u + L.d_wlen + 2u + L.pa[3] + 1u + L.d_glen + 1u;
  // "s " id pb0 pb1 " 0" pb2 " rlen S" pb3 " rlen " ROW "\n\n"
  L.readrow_rel = L.refrow_rel + ncol + 1u + 2u + L.idlen + L.pb_[0] + L.pb_[1] + 2u + L.pb_[2] + 1u + L.d_rlen + 2u +
                  L.pb_[3] + 1u + L.d_rlen + 1u;
  L.maf_size = L.readrow_rel + ncol + 2u;
  return L;
}

// record sizes and tile counts of every valid subread
__global__ void k_sizes(Batch B, EmitParams P, DeviceSet S, uint32_t n_sub, uint64_t *reads_size, uint64_t *maf_size,
                        uint64_t *ntiles, EmitLay *lay) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_sub) return;
  const uint32_t r = s / P.pass_num, pass = s % P.pass_num;
  const RefName N = ref_name(S, B, r, P.glen);
  const uint32_t shown = P.sample ? B.ncol[s] - B.nins[s] : B.plan_wlen[r];
  const RecLayout L = rec_layout(P, N, B.first_read + 1u + r, pass, shown, B.rlen[s], B.ncol[s]);
  reads_size[s] = L.reads_size;
  maf_size[s] = L.maf_size;
  EmitLay y;
  y.seq_rel = (uint32_t)L.seq_rel; y.qual_rel = (uint32_t)L.qual_rel; y.ip_rel = (uint32_t)L.ip_rel;
  y.pw_rel = (uint32_t)L.pw_rel; y.refrow_rel = (uint32_t)L.refrow_rel; y.readrow_rel = (uint32_t)L.readrow_rel;
  lay[s] = y;
  const uint32_t ne = B.nent[s];
  // segmented qshmm sub-reads: nent holds the tile count (errhmm tiles stay one contiguous stream)
  if (P.qs_segments && ((B.plan_meta[r] >> 11) & 1u)) ntiles[s] = ne == 0 ? 1u : ne;
  else ntiles[s] = ne == 0 ? 1u : (ne + PB_TILE - 1u) / PB_TILE;
}

__device__ __forceinline__ uint8_t *put_dec(uint8_t *p, uint64_t v, uint32_t nd) {
  for (uint32_t i = 0; i < nd; ++i) {
    p[nd - 1u - i] = (uint8_t)('0' + v % 10);
    v /= 10;
  }
  return p + nd;
}
__device__ __forceinline__ uint8_t *put_mem(uint8_t *p, const char *s, uint32_t n) {
  for (uint32_t i = 0; i < n; ++i) p[i] = (uint8_t)s[i];
  return p + n;
}
__device__ __forceinline__ uint8_t *put_pad(uint8_t *p, uint32_t n) {
  for (uint32_t i = 0; i < n; ++i) p[i] = ' ';
  return p + n;
}
#define PB_PUT_LIT(p, lit) put_mem((p), (lit), PB_LEN(lit))

__device__ __forceinline__ uint8_t *put_id(uint8_t *p, const EmitParams &P, uint64_t read_id, uint32_t pass,
                                           const RecLayout &L) {
  p = put_mem(p, P.id_head, P.id_head_len);
  if (!P.sam) {
    *p++ = '_';
    p = put_dec(p, read_id, L.d_rid);
  } else {
    *p++ = '/';
    p = put_dec(p, read_id, L.d_rid);
    *p++ = '/';
    p = put_dec(p, pass, L.d_pass);
  }
  return p;
}

// everything of a record that is not a per-base row: written once, by one lane
__device__ __noinline__ void write_headers(const EmitParams &P, const RefName &N, const RecLayout &L, uint8_t *rd,
                                           uint8_t *mf, uint64_t read_id, uint32_t pass, uint32_t wlen,
                                           uint32_t rlen, uint32_t ncol, uint32_t minus) {
  const uint32_t offset = N.off;
  uint8_t *p = rd;
  if (!P.sam) {
    *p++ = '@';
    p = put_id(p, P, read_id, pass, L);
    *p++ = '\n';
    p = rd + L.seq_rel + rlen;
    *p++ = '\n';
    *p++ = '+';
    p = put_id(p, P, read_id, pass, L);
    *p++ = '\n';
    rd[L.qual_rel + rlen] = '\n';
  } else if (P.sam == 2u) {
    auto put32 = [](uint8_t *q, uint32_t v) { q[0] = (uint8_t)v; q[1] = (uint8_t)(v >> 8); q[2] = (uint8_t)(v >> 16); q[3] = (uint8_t)(v >> 24); return q + 4; };
    auto put16 = [](uint8_t *q, uint32_t v) { q[0] = (uint8_t)v; q[1] = (uint8_t)(v >> 8); return q + 2; };
    auto put_int_tag = [&](uint8_t *q, char t0, char t1, int64_t v) {
      *q++ = (uint8_t)t0; *q++ = (uint8_t)t1; *q++ = bam_int_type(v);
      const uint32_t w = bam_int_width(v);
      for (uint32_t i = 0; i < w; ++i) *q++ = (uint8_t)((uint64_t)v >> (8u * i));
      return q;
    };
    p = put32(p, (uint32_t)(L.reads_size - 4u));  // block_size
    p = put32(p, 0xFFFFFFFFu);                    // refID -1
    p = put32(p, 0xFFFFFFFFu);                    // pos -1 (SAM POS 0)
    *p++ = (uint8_t)(L.idlen + 1u);               // l_read_name
    *p++ = 255;                                   // MAPQ
    p = put16(p, 4680u);                          // bin of an unmapped read: reg2bin(-1, 0)
    p = put16(p, 0u);                             // n_cigar_op
    p = put16(p, 4u);                             // FLAG: unmapped
    p = put32(p, rlen);                           // l_seq
    p = put32(p, 0xFFFFFFFFu);                    // next refID
    p = put32(p, 0xFFFFFFFFu);                    // next pos
    p = put32(p, 0u);                             // tlen
    p = put_id(p, P, read_id, pass, L);
    *p++ = 0;
    p = rd + L.qual_rel + rlen;
    *p++ = 'c'; *p++ = 'x'; *p++ = 'C'; *p++ = 3;
    *p++ = 'i'; *p++ = 'p'; *p++ = 'B'; *p++ = 'C';
    p = put32(p, rlen);
    p = rd + L.ip_rel + rlen;
    *p++ = 'n'; *p++ = 'p'; *p++ = 'C'; *p++ = 1;
    *p++ = 'p'; *p++ = 'w'; *p++ = 'B'; *p++ = 'C';
    p = put32(p, rlen);
    p = rd + L.tail_rel;
    *p++ = 'q'; *p++ = 's'; *p++ = 'C'; *p++ = 0;
    p = put_int_tag(p, 'q', 'e', (int64_t)rlen - 1);
    *p++ = 'r'; *p++ = 'q'; *p++ = 'f';
    p = put32(p, __float_as_uint(P.rq_f));
    *p++ = 's'; *p++ = 'n'; *p++ = 'B'; *p++ = 'f';
    p = put32(p, 4u);
    for (int i = 0; i < 4; ++i) p = put32(p, __float_as_uint(10.0f));
    p = put_int_tag(p, 'z', 'm', (int64_t)read_id);
    *p++ = 'R'; *p++ = 'G'; *p++ = 'Z';
    p = put_mem(p, "ffffffff", 8);
    *p++ = 0;
  } else {
    p = put_id(p, P, read_id, pass, L);
    p = PB_PUT_LIT(p, PB_SAM_S1);
    rd[L.seq_rel + rlen] = '\t';
    PB_PUT_LIT(rd + L.qual_rel + rlen, PB_SAM_S2);
    PB_PUT_LIT(rd + L.ip_rel + 2ull * rlen, PB_SAM_S3);
    p = rd + L.tail_rel;
    p = PB_PUT_LIT(p, PB_SAM_S4);
    if (rlen == 0) {
      *p++ = '-';
      *p++ = '1';
    } else {
      p = put_dec(p, rlen - 1u, ndigits(rlen - 1u));
    }
    p = PB_PUT_LIT(p, PB_SAM_S5);
    p = put_mem(p, P.rq, P.rq_len);
    p = PB_PUT_LIT(p, PB_SAM_S6);
    p = put_dec(p, read_id, L.d_rid);
    p = PB_PUT_LIT(p, PB_SAM_S7);
  }
  p = mf;
  p = PB_PUT_LIT(p, "a\ns ");
  if (N.ptr) p = put_mem(p, reinterpret_cast<const char *>(N.ptr), N.len);
  else p = PB_PUT_LIT(p, "ref");
  p = put_pad(p, L.pa[0] + L.pa[1]);
  *p++ = ' ';
  p = put_dec(p, offset, L.d_off);
  p = put_pad(p, L.pa[2]);
  *p++ = ' ';
  p = put_dec(p, wlen, L.d_wlen);
  *p++ = ' ';
  *p++ = '+';
  p = put_pad(p, L.pa[3]);
  *p++ = ' ';
  p = put_dec(p, N.src_len, L.d_glen);
  *p++ = ' ';
  p = mf + L.refrow_rel + ncol;
  *p++ = '\n';
  *p++ = 's';
  *p++ = ' ';
  p = put_id(p, P, read_id, pass, L);
  p = put_pad(p, L.pb_[0] + L.pb_[1]);
  *p++ = ' ';
  *p++ = '0';
  p = put_pad(p, L.pb_[2]);
  *p++ = ' ';
  p = put_dec(p, rlen, L.d_rlen);
  *p++ = ' ';
  *p++ = minus ? '-' : '+';
  p = put_pad(p, L.pb_[3]);
  *p++ = ' ';
  p = put_dec(p, rlen, L.d_rlen);
  *p++ = ' ';
  p = mf + L.readrow_rel + ncol;
  *p++ = '\n';
  *p++ = '\n';
}

__device__ __forceinline__ uint8_t comp_char(uint8_t c) {  // revcomp's complement (:5853-5863)
  switch (c) {
    case 'A': return 'T';
    case 'T': return 'A';
    case 'G': return 'C';
    case 'C': return 'G';
    default: return c;
  }
}

// reference bases of the generic tile path, from the ASCII copy of the genome
struct RefFetch {
  const uint8_t *__restrict__ ascii;
  uint32_t offset, wlen, minus;
  // window index r -> forward genome char, window-strand char, window-strand code, ACGT flag
  __device__ __forceinline__ void get(uint32_t r, uint8_t &gch, uint8_t &wch, uint32_t &wc, bool &acgt) const {
    const uint32_t g = minus ? offset + wlen - 1u - r : offset + r;
    const uint32_t lut = 0x54474341u;  // "ACGT"
    gch = __ldg(&ascii[g]);
    uint32_t gc = 0;
    acgt = true;
    switch (gch) {
      case 'A': gc = 0; break;
      case 'C': gc = 1; break;
      case 'G': gc = 2; break;
      case 'T': gc = 3; break;
      default: acgt = false; break;
    }
    wc = gc ^ (minus ? 3u : 0u);
    wch = acgt ? (uint8_t)(lut >> (8u * wc)) : gch;
  }
};

// read base from the event (window strand); substitution alphabets of set_mut (:5481-5486)
__device__ __forceinline__ uint8_t read_base(uint32_t kind, uint32_t info, uint8_t wch, uint32_t wc, bool acgt) {
  const uint32_t nt4 = 0x43475441u;  // "ATGC"
  if (kind == PB_KIND_MATCH) return wch;
  if (kind == PB_KIND_SUB) {
    if (!acgt) return (uint8_t)(nt4 >> (8u * (info & 3u)));
    // by window code A=0 C=1 G=2 T=3: A->"TGC" C->"ATG" G->"ATC" T->"AGC"
    const uint32_t subA = 0x00434754u, subC = 0x00475441u, subG = 0x00435441u, subT = 0x00434741u;
    const uint32_t tab = wc == 0u ? subA : (wc == 1u ? subC : (wc == 2u ? subG : subT));
    return (uint8_t)(tab >> (8u * (info > 2u ? 2u : info)));
  }
  // insertion: half of the time a copy of the current (not yet consumed) reference base (:2252-2257)
  return info >= 4u ? wch : (uint8_t)(nt4 >> (8u * info));
}

// ---- read-base codes of the staged tile path's lookup tables ------------------------------------
// Everything in 2-bit code space (A=0 C=1 G=2 T=3, complement = ^3), converted to characters with
// one byte-permute per output.  Substitution alphabets of set_mut (:5481-5486) as 2-bit codes:
//   A -> T,G,C   C -> A,T,G   G -> A,T,C   T -> A,G,C      index = window code * 3 + choice
__device__ __forceinline__ uint32_t sub_code(uint32_t wc, uint32_t choice) {
  // codes packed 2 bits each, entry (wc*3 + choice):  A:3,2,1  C:0,3,2  G:0,3,1  T:0,2,1
  const uint32_t tab = (3u) | (2u << 2) | (1u << 4) | (0u << 6) | (3u << 8) | (2u << 10) | (0u << 12) | (3u << 14) |
                       (1u << 16) | (0u << 18) | (2u << 20) | (1u << 22);
  return (tab >> ((wc * 3u + choice) * 2u)) & 3u;
}
// "ATGC"[i] (insertion alphabet, :5486) as a code: A T G C -> 0 3 2 1
__device__ __forceinline__ uint32_t ins_code(uint32_t i) { return (0x6Cu >> (i * 2u)) & 3u; }  // 0b01101100
__device__ __forceinline__ uint8_t code_char(uint32_t code) { return (uint8_t)__byte_perm(0x54474341u, 0u, code); }

// read-base code of an event given the window code of the current reference base
__device__ __forceinline__ uint32_t read_code(uint32_t kind, uint32_t info, uint32_t wc) {
  const uint32_t s = sub_code(wc, info > 2u ? 2u : info);
  const uint32_t i = info >= 4u ? wc : ins_code(info & 3u);
  return kind == PB_KIND_MATCH ? wc : (kind == PB_KIND_SUB ? s : i);
}

constexpr uint32_t kEmitPerLane = 4;                    // entries per lane per iteration
constexpr uint32_t kEmitStep = 32u * kEmitPerLane;      // entries per warp iteration

// Everything the row kernel needs to know about a tile, gathered once by k_tile_desc (one THREAD per tile: the
// dependent loads through tile -> sub-read -> plan / layout / checkpoints run with full memory-level parallelism
// there instead of as a serial prologue in front of every tile).
struct TileDesc {
  uint64_t ev_off;          // byte offset of the tile's first entry in the event arena
  uint64_t o_seq, o_qual;   // byte offsets in the reads stream of the tile's first read base / quality (BAM: o_seq
                            // is the nibble offset of the base, two per byte, high nibble first)
  uint64_t o_ref, o_read;   // byte offsets in the MAF stream of the tile's first column (file order) in both rows
  uint32_t e1;              // entries of the tile
  uint32_t Pn, Cn, Rn;      // read bases, MAF columns and window bases it covers
  uint32_t wpos;            // genome index of the tile's first window base (the minus strand walks down from it)
  uint32_t flags;           // kTile*
};
static_assert(sizeof(TileDesc) == 64, "four 16-byte loads");
constexpr uint32_t kTileMinus = 1u, kTileGeneric = 2u, kTileWide = 4u, kTileEmpty = 8u;

// ---- staged tile path -----------------------------------------------------------------------
// The four per-base rows of a tile (read bases, qualities, MAF reference row, MAF read row) are contiguous
// fragments of the records (the MAF fragments of a minus-strand read run backwards, but they are still one
// range each).  The warp builds them in shared memory and then copies every fragment to HBM with 16-byte
// stores: the staging buffer of a row starts at the same offset modulo 16 as its destination, so aligned
// chunks of the record are aligned chunks of the buffer; only the first and last chunk of a fragment (shared
// with the neighbouring tiles) are written bytewise.  The window bases of the tile are staged first as 2-bit
// codes in WINDOW order (reversed and complemented for the minus strand), so a lane gets the 16 bases that
// follow its first entry with two shared-memory loads and a funnel shift.
constexpr uint32_t kStageCols = 1280;   // MAF columns a tile may have on this path (more: direct path)
struct EmitStage {
  uint8_t seq[PB_TILE + 32];
  uint8_t qual[PB_TILE + 32];
  uint8_t mref[kStageCols + 80];   // rows end before + 32; bytes + 48 .. + 79: one scratch byte per lane
  uint8_t mread[kStageCols + 80];
  uint32_t pk[kStageCols / 16 + 8];
};
static_assert(sizeof(EmitStage) % 16 == 0, "staging rows stay 16-byte aligned");

// window codes of the 16 window positions from tile-relative position r on (2 bits each, position r in bits 0-1);
// wpos: genome index of the tile's window position 0
__device__ __forceinline__ uint32_t window_word(const uint32_t *__restrict__ pk, uint32_t wpos, uint32_t minus,
                                                uint32_t glen_words, uint32_t r) {
  // plus strand: genome positions wpos + r .. + 15; minus strand: wpos - r - 15 .. wpos - r, reversed and complemented
  const int64_t gl = minus ? (int64_t)wpos - (int64_t)r - 15 : (int64_t)wpos + (int64_t)r;
  uint32_t x;
  if (gl >= 0) {
    const uint32_t g = (uint32_t)gl;
    const uint32_t w = g >> 4, sh = (g & 15u) * 2u;
    const uint32_t lo = __ldg(&pk[w]);
    const uint32_t hi = (w + 1u < glen_words) ? __ldg(&pk[w + 1u]) : 0u;
    x = __funnelshift_r(lo, hi, sh);
  } else {
    if (gl < -15) return 0u;                                             // wholly in front of the genome (never read)
    x = __ldg(&pk[0]) << (uint32_t)(-gl * 2);                            // genome positions 0 .. in the top fields
  }
  if (!minus) return x;
  x = __brev(x);                                                         // reverse the 16 fields ...
  x = ((x & 0x55555555u) << 1) | ((x >> 1) & 0x55555555u);               // ... keeping the bit order inside a field
  return ~x;                                                             // complement: code ^ 3
}

// copy `n` staged bytes to g; buf[shift + i] holds byte i and (g - shift) is 16-byte aligned.  Whole 16-byte
// chunks go out as vectors; the bytes of the partial first and last chunk one per lane.
__device__ __forceinline__ void flush_row(const uint8_t *buf, uint8_t *__restrict__ g, uint32_t n, uint32_t shift,
                                          uint32_t lane) {
  const uint32_t total = shift + n;
  uint8_t *g0 = g - shift;
  const uint32_t body_lo = shift ? 16u : 0u, body_hi = total & ~15u;   // [body_lo, body_hi): whole chunks (if any)
  for (uint32_t lo = body_lo + lane * 16u; lo < body_hi; lo += 512u)
    *reinterpret_cast<uint4 *>(g0 + lo) = *reinterpret_cast<const uint4 *>(buf + lo);
  const uint32_t head_end = shift ? (total < 16u ? total : 16u) : 0u;  // head: bytes [shift, head_end)
  uint32_t tail_start = body_hi > body_lo ? body_hi : body_lo;         // tail: bytes [tail_start, total)
  if (tail_start < head_end) tail_start = head_end;
  if (shift + lane < head_end) g0[shift + lane] = buf[shift + lane];
  if (tail_start + lane < total) g0[tail_start + lane] = buf[tail_start + lane];
}

// 8 BAM base codes, one per byte of x and y -> 4 bytes of two bases each (high nibble first); codes outside the
// tile are whatever the staging row held, hence the masks
__device__ __forceinline__ uint32_t pack_codes(uint32_t x, uint32_t y) {
  x &= 0x0F0F0F0Fu;
  y &= 0x0F0F0F0Fu;
  return __byte_perm((x << 4) | (x >> 8), (y << 4) | (y >> 8), 0x6420u);
}

// BAM read bases: buf[shift + i] holds the code of base i, g0 the 16-byte aligned byte whose high nibble is buf[0].
// The codes are packed two per byte in place; the bytes that hold two bases of the tile go out through flush_row, a
// first / last byte that the tile shares with its neighbour (odd start / end) gets its nibble with an atomic OR
// into the zeroed record.
__device__ __forceinline__ void flush_nibbles(uint8_t *buf, uint8_t *__restrict__ g0, uint32_t n, uint32_t shift,
                                              uint32_t lane) {
  if (n == 0u) return;
  const uint32_t total = shift + n;
  for (uint32_t j0 = 0; j0 < total; j0 += 1024u) {  // 32 codes per lane -> 16 bytes, written over codes already read
    const uint32_t j = j0 + lane * 32u;
    uint4 a = make_uint4(0u, 0u, 0u, 0u), b = a;
    if (j < total) {
      a = *reinterpret_cast<const uint4 *>(buf + j);
      b = *reinterpret_cast<const uint4 *>(buf + j + 16u);
    }
    __syncwarp();
    if (j < total)
      *reinterpret_cast<uint4 *>(buf + j / 2u) =
          make_uint4(pack_codes(a.x, a.y), pack_codes(a.z, a.w), pack_codes(b.x, b.y), pack_codes(b.z, b.w));
  }
  __syncwarp();
  const uint32_t lo = (shift + 1u) >> 1, hi = total >> 1;  // bytes [lo, hi) hold two bases of the tile
  flush_row(buf + (lo & ~15u), g0 + lo, hi - lo, lo & 15u, lane);
  if (lane == 0u && (shift & 1u)) atomic_or_byte(g0 + (shift >> 1), buf[shift >> 1] & 0x0Fu);
  if (lane == 1u && (total & 1u)) atomic_or_byte(g0 + (total >> 1), buf[total >> 1] & 0xF0u);
}

// byte LUTs of the staged path, index = (kind | info << 2) << 2 | window code of the current reference base
// (kind 3 = errhmm deletion column).  seq: the read base (BAM: its 4-bit code 1 << code); mread / mref: the MAF
// characters for the plus ([0]) and the minus strand ([1], complemented because the rows are mirrored back).
struct EmitLuts {
  uint8_t seq[128];
  uint8_t mread[2][128];
  uint8_t mref[2][128];
};
template <bool BAM>
__device__ __forceinline__ void build_emit_luts(EmitLuts &L, uint32_t t) {  // t = 0 .. 127
  const uint32_t wc = t & 3u, kind = (t >> 2) & 3u, info = (t >> 4) & 7u;
  const uint32_t rc = read_code(kind == 3u ? 0u : kind, info, wc);
  L.seq[t] = BAM ? (uint8_t)(1u << rc) : code_char(rc);
  for (uint32_t f = 0; f < 2u; ++f) {
    const uint32_t flip = f ? 3u : 0u;
    L.mread[f][t] = kind == 3u ? (uint8_t)'-' : code_char(rc ^ flip);
    L.mref[f][t] = kind == PB_KIND_INS ? (uint8_t)'-' : code_char(wc ^ flip);
  }
}

// One tile whose reference range holds only ACGT (Cn <= kStageCols, Pn <= PB_TILE).  BAM: g_seq is the byte of the
// tile's first base, seq_odd 1 when that base is its low nibble; qualities are the values themselves.
template <int METHOD, bool BAM>
__device__ __forceinline__ void emit_tile_staged(EmitStage &S, const EmitLuts &LU, const uint8_t *__restrict__ evbase,
                                                 uint32_t e1, const uint32_t *__restrict__ pk, uint32_t glen_words,
                                                 uint32_t wpos, uint32_t minus, uint32_t Pn, uint32_t Cn, uint32_t Rn,
                                                 uint8_t *__restrict__ g_seq, uint32_t seq_odd, uint8_t *__restrict__ g_qual,
                                                 uint8_t *__restrict__ g_ref, uint8_t *__restrict__ g_read, uint32_t lane) {
  const uint32_t e0 = 0;
  constexpr uint32_t qoff = BAM ? 0u : 33u;  // '!' + quality value
  // the offsets (modulo 16) the staging rows of the four fragments start at; BAM bases: the nibble offset modulo 32
  const uint32_t sh_s = BAM ? 2u * (uint32_t)(reinterpret_cast<uintptr_t>(g_seq) & 15u) + seq_odd
                            : (uint32_t)(reinterpret_cast<uintptr_t>(g_seq) & 15u);
  const uint32_t sh_q = (uint32_t)(reinterpret_cast<uintptr_t>(g_qual) & 15u);
  const uint32_t sh_r = (uint32_t)(reinterpret_cast<uintptr_t>(g_ref) & 15u);
  const uint32_t sh_m = (uint32_t)(reinterpret_cast<uintptr_t>(g_read) & 15u);
  // staging indices: column c of the tile lives at S.mref[o_ref + c * cdir] (the minus strand's rows run backwards)
  const int32_t cdir = minus ? -1 : 1;
  const uint32_t o_ref = sh_r + (minus ? Cn - 1u : 0u);
  const uint32_t d_read = sh_m - sh_r;                           // S.mread index of a column = its S.mref index + d_read (mod 2^32)
  const uint32_t o_dump = kStageCols + 48u + lane;               // this lane's scratch byte behind the rows
  const uint32_t moff = minus ? 128u : 0u;                       // strand half of the MAF character LUTs
  const uint32_t ref_chars = minus ? 0x41434754u : 0x54474341u;  // "TGCA" / "ACGT": MAF character of a window code
  // the MAF read row starts as all '-': deletion columns then only need their reference character
  for (uint32_t j = lane * 16u; j < sh_m + Cn; j += 512u)
    *reinterpret_cast<uint4 *>(S.mread + j) = make_uint4(0x2D2D2D2Du, 0x2D2D2D2Du, 0x2D2D2D2Du, 0x2D2D2D2Du);
  // ---- window codes of the tile: positions R0 .. R0 + Rn (an insertion at the end looks at R0 + Rn) + 16 spare
  const uint32_t nw = (Rn + 16u) / 16u + 1u;
  for (uint32_t j = lane; j < nw; j += 32u) S.pk[j] = window_word(pk, wpos, minus, glen_words, 16u * j);
  __syncwarp();
  auto load_entries = [&](uint32_t i) -> uint2 {
    const uint32_t eb = i + lane * kEmitPerLane;
    if (METHOD == PBSIM_METHOD_QSHMM) return __ldg(reinterpret_cast<const uint2 *>(evbase + 2ull * eb));
    return make_uint2(__ldg(reinterpret_cast<const uint32_t *>(evbase + eb)), 0u);
  };
  auto codes_at = [&](uint32_t r) -> uint32_t {   // the 16 window bases from tile-relative position r on
    return __funnelshift_r(S.pk[r >> 4], S.pk[(r >> 4) + 1u], (r & 15u) * 2u);
  };
  uint32_t Pt = 0, Rt = 0, Ct = 0;   // tile-relative totals so far
  uint2 nxt = load_entries(e0);
  for (uint32_t i = e0; i < e1; i += kEmitStep) {
    const uint32_t eb = i + lane * kEmitPerLane;
    const uint2 v = nxt;
    if (i + kEmitStep < e1) nxt = load_entries(i + kEmitStep);
    uint32_t raw[kEmitPerLane];
    if (METHOD == PBSIM_METHOD_QSHMM) {
      raw[0] = v.x & 0xFFFFu; raw[1] = v.x >> 16; raw[2] = v.y & 0xFFFFu; raw[3] = v.y >> 16;
    } else {
      raw[0] = v.x & 0xFFu; raw[1] = (v.x >> 8) & 0xFFu; raw[2] = (v.x >> 16) & 0xFFu; raw[3] = v.x >> 24;
    }
    // common case: 128 valid entries, none of them a continuation entry, no lane with more than 11 deletions
    // (so the 16 window bases a lane fetches cover everything its four entries touch)
    uint32_t li = 0, ld = 0;
    uint32_t idx[kEmitPerLane], nd[kEmitPerLane];
#pragma unroll
    for (uint32_t k = 0; k < kEmitPerLane; ++k) {
      if (METHOD == PBSIM_METHOD_QSHMM) {
        idx[k] = (raw[k] >> 5) & 0x7Cu;       // (kind | info << 2) << 2
        nd[k] = raw[k] >> 12;
        li += (raw[k] >> 8) & 1u;             // kind 2
      } else {
        idx[k] = (raw[k] & 0x1Fu) << 2;
        nd[k] = ((raw[k] & 3u) == PB_KIND_DEL) ? 1u : 0u;
        li += ((raw[k] & 3u) == PB_KIND_INS) ? 1u : 0u;
      }
      ld += nd[k];
    }
    bool plain = i + kEmitStep <= e1;
    if (METHOD == PBSIM_METHOD_QSHMM) {
      const uint32_t cont = ((v.x & (v.x >> 1)) | (v.y & (v.y >> 1))) & 0x00800080u;  // kind == 3 in one of the four
      plain = plain && !__any_sync(0xFFFFFFFFu, (cont != 0u) || (ld > 11u));
    }
    if (plain) {
      const uint32_t mine = li | (ld << 8);     // <= 128 insertions, <= 12 * 32 deletions per iteration
      uint32_t x = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= (uint32_t)o) x += y;
      }
      const uint32_t tot = __shfl_sync(0xFFFFFFFFu, x, 31);
      const uint32_t pre = x - mine;
      const uint32_t pre_i = pre & 0xFFu, pre_d = pre >> 8;
      uint32_t Pp, Rr, Cc;
      if (METHOD == PBSIM_METHOD_QSHMM) {       // an entry is a read base (+ deletions behind it)
        Pp = Pt + lane * kEmitPerLane;
        Rr = Rt + lane * kEmitPerLane - pre_i + pre_d;
        Cc = Ct + lane * kEmitPerLane + pre_d;
      } else {                                  // an entry is an alignment column
        Cc = Ct + lane * kEmitPerLane;
        Rr = Rt + lane * kEmitPerLane - pre_i;
        Pp = Pt + lane * kEmitPerLane - pre_d;
      }
      uint32_t bits = codes_at(Rr);             // consumed two bits at a time as the reference advances
      // 32-bit staging indices (generic 64-bit pointers into shared memory cost two instructions per step)
      uint32_t oc = o_ref + Cc * (uint32_t)cdir;   // this column's byte in S.mref; S.mread: + d_read
      if (METHOD == PBSIM_METHOD_QSHMM) {
        const uint32_t op = Pp;
        uint32_t multi = 0;
        const uint32_t bits0 = bits, oc0 = oc;
#pragma unroll
        for (uint32_t k = 0; k < kEmitPerLane; ++k) {
          const uint32_t t = idx[k] | (bits & 3u);
          S.seq[sh_s + op + k] = LU.seq[t];
          S.qual[sh_q + op + k] = (uint8_t)((raw[k] & 0x7Fu) + qoff);
          S.mread[oc + d_read] = LU.mread[0][t + moff];
          S.mref[oc] = LU.mref[0][t + moff];
          oc += (uint32_t)cdir;
          if (!(raw[k] & 0x100u)) bits >>= 2;   // an insertion does not consume the reference base
          // deleted reference bases behind the entry: the read row already holds '-' (prefilled); the first
          // deleted base is stored without a branch (to a scratch byte when there is none)
          const uint32_t dst = nd[k] ? oc : o_dump;
          S.mref[dst] = (uint8_t)__byte_perm(ref_chars, 0u, bits & 3u);
          multi |= nd[k];
          oc += nd[k] * (uint32_t)cdir;
          bits >>= 2u * nd[k];
        }
        if (multi > 1u) {   // an entry with two or more deletions (rare): their further reference characters
          uint32_t b2 = bits0, o2 = oc0;
#pragma unroll
          for (uint32_t k = 0; k < kEmitPerLane; ++k) {
            o2 += (uint32_t)cdir;
            if (!(raw[k] & 0x100u)) b2 >>= 2;
            for (uint32_t j = 1; j < nd[k]; ++j)
              S.mref[o2 + j * (uint32_t)cdir] = (uint8_t)__byte_perm(ref_chars, 0u, (b2 >> (2u * j)) & 3u);
            o2 += nd[k] * (uint32_t)cdir;
            b2 >>= 2u * nd[k];
          }
        }
      } else {
        uint32_t op = Pp;
#pragma unroll
        for (uint32_t k = 0; k < kEmitPerLane; ++k) {
          const uint32_t t = idx[k] | (bits & 3u);
          const bool isb = nd[k] == 0u;
          if (isb) {
            S.seq[sh_s + op] = LU.seq[t];
            S.qual[sh_q + op] = (uint8_t)qoff;
          }
          S.mread[oc + d_read] = LU.mread[0][t + moff];
          S.mref[oc] = LU.mref[0][t + moff];
          oc += (uint32_t)cdir;
          op += isb ? 1u : 0u;
          if ((raw[k] & 3u) != PB_KIND_INS) bits >>= 2;
        }
      }
      const uint32_t tot_i = tot & 0xFFu, tot_d = tot >> 8;
      if (METHOD == PBSIM_METHOD_QSHMM) {
        Pt += kEmitStep; Rt += kEmitStep - tot_i + tot_d; Ct += kEmitStep + tot_d;
      } else {
        Ct += kEmitStep; Rt += kEmitStep - tot_i; Pt += kEmitStep - tot_d;
      }
      continue;
    }
    // ---- general iteration: entries past the end of the tile, continuation entries
    uint32_t kind[kEmitPerLane], info[kEmitPerLane], isb[kEmitPerLane], adv[kEmitPerLane];
    uint32_t lb = 0, la = 0;
    ld = 0;
#pragma unroll
    for (uint32_t k = 0; k < kEmitPerLane; ++k) {
      const bool valid = eb + k < e1;
      const uint32_t x = raw[k];
      if (METHOD == PBSIM_METHOD_QSHMM) {
        kind[k] = (x >> 7) & 3u;
        info[k] = (x >> 9) & 7u;
        const bool cont = kind[k] == 3u;
        nd[k] = valid ? (cont ? ((x & 0x7Fu) | ((x >> 9) << 7)) : (x >> 12)) : 0u;
        isb[k] = (valid && !cont) ? 1u : 0u;
      } else {
        kind[k] = x & 3u;
        info[k] = (x >> 2) & 7u;
        nd[k] = (valid && kind[k] == PB_KIND_DEL) ? 1u : 0u;
        isb[k] = (valid && kind[k] != PB_KIND_DEL) ? 1u : 0u;
      }
      adv[k] = (isb[k] && kind[k] != PB_KIND_INS) ? 1u : 0u;
      lb += isb[k];
      la += adv[k];
      ld += nd[k];
    }
    // one warp scan over the packed per-lane totals: bases (8 bit) | advances (8 bit) | deletions (16 bit);
    // Cn <= kStageCols bounds every count of the tile, so the packed fields cannot overflow
    const uint32_t mine = lb | (la << 8) | (ld << 16);
    uint32_t x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (uint32_t)o) x += y;
    }
    const uint32_t tot = __shfl_sync(0xFFFFFFFFu, x, 31);
    const uint32_t pre = x - mine;
    uint32_t Pp = Pt + (pre & 0xFFu), Rr = Rt + ((pre >> 8) & 0xFFu) + (pre >> 16), Cc = Ct + (pre & 0xFFu) + (pre >> 16);
    for (uint32_t k = 0; k < kEmitPerLane; ++k) {
      if (isb[k]) {
        const uint32_t t = ((kind[k] | (info[k] << 2)) << 2) | (codes_at(Rr) & 3u);
        S.seq[sh_s + Pp] = LU.seq[t];
        S.qual[sh_q + Pp] = METHOD == PBSIM_METHOD_QSHMM ? (uint8_t)((raw[k] & 0x7Fu) + qoff) : (uint8_t)qoff;
        S.mread[o_ref + Cc * (uint32_t)cdir + d_read] = LU.mread[0][t + moff];
        S.mref[o_ref + Cc * (uint32_t)cdir] = LU.mref[0][t + moff];
        ++Pp;
        ++Cc;
        Rr += adv[k];
      }
      for (uint32_t j = 0; j < nd[k]; ++j) {
        S.mread[o_ref + Cc * (uint32_t)cdir + d_read] = '-';
        S.mref[o_ref + Cc * (uint32_t)cdir] = LU.mref[0][(codes_at(Rr) & 3u) + moff];
        ++Cc;
        ++Rr;
      }
    }
    Pt += tot & 0xFFu;
    Rt += ((tot >> 8) & 0xFFu) + (tot >> 16);
    Ct += (tot & 0xFFu) + (tot >> 16);
  }
  __syncwarp();
  if (BAM) flush_nibbles(S.seq, g_seq - (sh_s >> 1), Pn, sh_s, lane);
  else flush_row(S.seq, g_seq, Pn, sh_s, lane);
  flush_row(S.qual, g_qual, Pn, sh_q, lane);
  flush_row(S.mref, g_ref, Cn, sh_r, lane);
  flush_row(S.mread, g_read, Cn, sh_m, lane);
  __syncwarp();
}

// generic tile path: reads the ASCII copy where the tile touches non-ACGT bases; one entry per lane
template <int METHOD, bool BAM>
__device__ __noinline__ void emit_tile_generic(const uint8_t *evbase, uint32_t e0, uint32_t e1, const RefFetch &rf,
                                               uint32_t minus, uint32_t ncol, uint32_t C0, uint32_t R0, uint32_t P0,
                                               uint8_t *seq, uint8_t *qual, uint8_t *mref, uint8_t *mread,
                                               uint32_t lane, const PhiloxKeys *keys, uint32_t read_id, uint32_t pass) {
  const uint32_t lt_mask = (1u << lane) - 1u;
  for (uint32_t i = e0; i < e1; i += 32u) {
    const uint32_t e = i + lane;
    const bool valid = e < e1;
    uint32_t kind = 0, info = 0, qv = 0, nd = 0;
    bool isbase = false;
    if (METHOD == PBSIM_METHOD_QSHMM) {
      const uint32_t v = valid ? (uint32_t)__ldg(reinterpret_cast<const uint16_t *>(evbase) + e) : 0u;
      kind = (v >> 7) & 3u;
      const bool cont = valid && kind == 3u;
      qv = v & 0x7Fu;
      info = (v >> 9) & 7u;
      nd = cont ? ((v & 0x7Fu) | ((v >> 9) << 7)) : ((v >> 12) & 15u);
      if (!valid) nd = 0;
      isbase = valid && !cont;
    } else {
      const uint32_t v = valid ? (uint32_t)__ldg(evbase + e) : 0u;
      kind = v & 3u;
      info = (v >> 2) & 7u;
      isbase = valid && kind != PB_KIND_DEL;
      nd = (valid && kind == PB_KIND_DEL) ? 1u : 0u;
    }
    const bool adv = isbase && kind != PB_KIND_INS;
    const uint32_t m_base = __ballot_sync(0xFFFFFFFFu, isbase);
    const uint32_t m_adv = __ballot_sync(0xFFFFFFFFu, adv);
    uint32_t x = nd;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (uint32_t)o) x += y;
    }
    const uint32_t tot_d = __shfl_sync(0xFFFFFFFFu, x, 31);
    const uint32_t pre_d = x - nd;
    const uint32_t Pp = P0 + __popc(m_base & lt_mask);
    const uint32_t Rr = R0 + __popc(m_adv & lt_mask) + pre_d;
    const uint32_t Cc = C0 + __popc(m_base & lt_mask) + pre_d;
    if (isbase) {
      uint8_t gch, wch;
      uint32_t wc;
      bool acgt;
      rf.get(Rr, gch, wch, wc, acgt);
      if (keys != nullptr && kind == PB_KIND_SUB && !acgt) {
        // PHILOX mode: the 4-way choice of this position, re-derived from its own draws (sim_core.cuh: qshmm /
        // sample bits 3-4 of word Y of read position Pp; errhmm bits 12-13 of word 0 of alignment column Cc)
        if (METHOD == PBSIM_METHOD_QSHMM) {
          uint32_t x, y;
          error_words_at(*keys, read_id, pass << 16, Pp, x, y);
          info = (y >> 3) & 3u;
        } else {
          uint32_t w[4];
          philox_block_keys(*keys, Cc, pass << 16, read_id, 1u, w);
          info = (w[0] >> 12) & 3u;
        }
      }
      const uint8_t rb = read_base(kind, info, wch, wc, acgt);
      put_read_base<BAM>(seq, qual, Pp, rb, BAM ? bam_nibble(rb) : 0u, qv, METHOD == PBSIM_METHOD_QSHMM);
      const uint32_t col = minus ? ncol - 1u - Cc : Cc;
      mread[col] = minus ? comp_char(rb) : rb;
      mref[col] = (kind == PB_KIND_INS) ? (uint8_t)'-' : gch;
    }
    if (nd != 0u) {
      const uint32_t cbase = Cc + (isbase ? 1u : 0u);
      const uint32_t rbase = Rr + (adv ? 1u : 0u);
      for (uint32_t j = 0; j < nd; ++j) {
        uint8_t gch, wch;
        uint32_t wc;
        bool acgt;
        rf.get(rbase + j, gch, wch, wc, acgt);
        const uint32_t col = minus ? ncol - 1u - (cbase + j) : cbase + j;
        mread[col] = '-';
        mref[col] = gch;
      }
    }
    P0 += __popc(m_base);
    R0 += __popc(m_adv) + tot_d;
    C0 += __popc(m_base) + tot_d;
  }
}

// what a tile covers, from the sub-read's arrays and checkpoints (shared by k_tile_desc and k_emit)
struct TileGeom {
  uint32_t e0, e1, has_next, Rnext, Pn, Cn, segmented, slow;
  Ckpt c0;
};
template <int METHOD>
__device__ __forceinline__ TileGeom tile_geom(const EmitArgs &A, uint32_t s, uint32_t r, uint32_t tile, uint32_t nent,
                                              uint32_t rlen, uint32_t ncol, uint32_t offset, uint32_t wlen, uint32_t minus) {
  TileGeom g;
  const Ckpt *ckp = A.ck + A.B.ck_off[s];
  g.c0 = ckp[tile];
  // sequential pass 1: one contiguous stream, tile = entries [1024 t, 1024 (t+1)); segment-parallel pass 1:
  // tile t lives in its own slot (stride PB_SEG_STRIDE) and its entry count is in the checkpoint
  g.segmented = (METHOD == PBSIM_METHOD_QSHMM && ((A.B.plan_meta[r] >> 11) & 1u)) ? 1u : 0u;
  g.e0 = g.segmented ? 0u : tile * PB_TILE;
  g.e1 = g.segmented ? g.c0.pad : min(nent, g.e0 + PB_TILE);
  g.has_next = (g.segmented ? (tile + 1u < nent) : (g.e1 < nent)) ? 1u : 0u;
  // reference range this tile can touch: [R0, Rend] (an insertion at the tile's end looks at Rend)
  Ckpt c1 = g.c0;
  if (g.has_next) c1 = ckp[tile + 1];
  // (--method sample: a read that is as long as its quality string ends with window bases left over, :1775-1833;
  // the reference bases it consumed are its columns minus its insertions)
  g.Rnext = g.has_next ? c1.ref : (A.P.sample ? min(wlen, ncol - A.B.nins[s]) : wlen);
  const uint32_t Rend = min(g.Rnext, wlen - 1u);
  const uint32_t g0 = minus ? offset + wlen - 1u - Rend : offset + g.c0.ref;
  const uint32_t g1 = minus ? offset + wlen - 1u - g.c0.ref : offset + Rend;
  g.slow = range_exceptional(A.G.xm, g0, g1) ? 1u : 0u;
  // what the tile covers: read bases, MAF columns (up to the next tile's checkpoint / the read's end)
  g.Pn = (g.has_next ? c1.read : rlen) - g.c0.read;
  g.Cn = (g.has_next ? c1.col : ncol) - g.c0.col;
  return g;
}

// One THREAD per tile: its sub-read (largest s with tile_start[s] <= t) and its descriptor.
template <int METHOD>
__global__ void k_tile_desc(const __grid_constant__ EmitArgs A, uint32_t *tile_sub) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= A.n_tiles) return;
  uint32_t lo = 0, hi = A.n_sub;
  while (hi - lo > 1u) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(&A.tile_start[mid]) <= t) lo = mid; else hi = mid;
  }
  const uint32_t s = lo;
  tile_sub[t] = s;
  const uint32_t tile = (uint32_t)(t - __ldg(&A.tile_start[s]));
  const uint32_t r = s / A.P.pass_num;
  const uint32_t offset = A.B.plan_off[r], wlen = A.B.plan_wlen[r];
  const uint32_t minus = (A.B.plan_meta[r] >> 8) & 1u;
  const uint32_t nent = A.B.nent[s], rlen = A.B.rlen[s], ncol = A.B.ncol[s];
  TileDesc d;
  memset(&d, 0, sizeof d);
  if (nent == 0) {
    d.flags = kTileEmpty;
  } else {
    const TileGeom g = tile_geom<METHOD>(A, s, r, tile, nent, rlen, ncol, offset, wlen, minus);
    const EmitLay L = A.lay[s];
    const uint64_t rd = A.reads_off[s], mf = A.maf_off[s];
    d.ev_off = (A.B.ev_off[s] + (g.segmented ? (uint64_t)tile * PB_SEG_STRIDE : (uint64_t)g.e0)) *
               (METHOD == PBSIM_METHOD_QSHMM ? 2ull : 1ull);
    d.o_seq = A.P.sam == 2u ? 2ull * (rd + L.seq_rel) + g.c0.read : rd + L.seq_rel + g.c0.read;
    d.o_qual = rd + L.qual_rel + g.c0.read;
    const uint32_t cfirst = minus ? ncol - g.c0.col - g.Cn : g.c0.col;   // first MAF column (file order) of the tile
    d.o_ref = mf + L.refrow_rel + cfirst;
    d.o_read = mf + L.readrow_rel + cfirst;
    d.e1 = g.e1 - g.e0;
    d.Pn = g.Pn;
    d.Cn = g.Cn;
    d.Rn = g.Rnext - g.c0.ref;
    d.wpos = minus ? offset + wlen - 1u - g.c0.ref : offset + g.c0.ref;
    d.flags = (minus ? kTileMinus : 0u) | (g.slow ? kTileGeneric : 0u) |
              ((g.Cn > kStageCols || g.Pn > PB_TILE || d.Rn > kStageCols) ? kTileWide : 0u);
  }
  uint4 *dst = reinterpret_cast<uint4 *>(A.desc + t);
  const uint4 *src = reinterpret_cast<const uint4 *>(&d);
  dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
}

// The ROW kernel of pass 2 (text and BAM records): one warp per tile, everything it needs in the tile's descriptor.
// Tiles that touch exceptional bases or are too wide for the staging rows are left to k_emit, as are the record
// headers and the SAM ip / pw arrays.  Kept small on purpose: the loop must live in the instruction cache.
template <int METHOD, bool BAM>
__global__ void __launch_bounds__(kEmitThreads, 4) k_emit_rows(const TileDesc *__restrict__ desc, uint64_t n_tiles,
                                                              const uint8_t *__restrict__ ev,
                                                              const uint32_t *__restrict__ pk, uint32_t glen_words,
                                                              uint8_t *__restrict__ out_reads,
                                                              uint8_t *__restrict__ out_maf) {
  __shared__ __align__(16) EmitStage stage[kEmitWarps];
  __shared__ EmitLuts luts;
  if (threadIdx.x < 128u) build_emit_luts<BAM>(luts, threadIdx.x);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warp0 = (uint64_t)blockIdx.x * kEmitWarps + (threadIdx.x >> 5);
  const uint64_t nwarps = (uint64_t)gridDim.x * kEmitWarps;
  for (uint64_t t = warp0; t < n_tiles; t += nwarps) {
    const uint4 *dp = reinterpret_cast<const uint4 *>(desc + t);
    const uint4 d0 = __ldg(dp), d1 = __ldg(dp + 1), d2 = __ldg(dp + 2), d3 = __ldg(dp + 3);
    const uint32_t flags = d3.w;
    if (flags & (kTileGeneric | kTileWide | kTileEmpty)) continue;
    const uint64_t ev_off = (uint64_t)d0.x | ((uint64_t)d0.y << 32), o_seq = (uint64_t)d0.z | ((uint64_t)d0.w << 32);
    const uint64_t o_qual = (uint64_t)d1.x | ((uint64_t)d1.y << 32), o_ref = (uint64_t)d1.z | ((uint64_t)d1.w << 32);
    const uint64_t o_read = (uint64_t)d2.x | ((uint64_t)d2.y << 32);
    emit_tile_staged<METHOD, BAM>(stage[threadIdx.x >> 5], luts, ev + ev_off, d2.z /* e1 */, pk, glen_words,
                                  d3.z /* wpos */, flags & kTileMinus, d2.w /* Pn */, d3.x /* Cn */, d3.y /* Rn */,
                                  out_reads + (BAM ? o_seq >> 1 : o_seq), BAM ? (uint32_t)o_seq & 1u : 0u,
                                  out_reads + o_qual, out_maf + o_ref, out_maf + o_read, lane);
  }
}

// Everything of pass 2 that is not a staged tile: the record headers (once per sub-read), tiles that touch
// exceptional bases or are too wide for the staging rows, and the SAM / BAM ip / pw arrays.
template <int METHOD, bool BAM>
__global__ void __launch_bounds__(kEmitThreads) k_emit(const __grid_constant__ EmitArgs A) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warp0 = (uint64_t)blockIdx.x * kEmitWarps + (threadIdx.x >> 5);
  const uint64_t nwarps = (uint64_t)gridDim.x * kEmitWarps;
  for (uint64_t t = warp0; t < A.n_tiles; t += nwarps) {
    const uint32_t s = __ldg(&A.tile_sub[t]);
    const uint32_t tile = (uint32_t)(t - __ldg(&A.tile_start[s]));
    // tiles the row kernel handles: nothing to do here unless the tile opens a record or SAM / BAM arrays follow
    const uint32_t dflags = __ldg(&A.desc[t].flags);
    const bool rows_here = (dflags & (kTileGeneric | kTileWide)) != 0u;
    if (!rows_here && tile != 0u && !A.P.sam) continue;
    const uint32_t r = s / A.P.pass_num, pass = s % A.P.pass_num;
    const uint64_t read_id = A.B.first_read + 1u + r;
    const uint32_t offset = A.B.plan_off[r], wlen = A.B.plan_wlen[r];
    const uint32_t minus = (A.B.plan_meta[r] >> 8) & 1u;
    const uint32_t nent = A.B.nent[s], rlen = A.B.rlen[s], ncol = A.B.ncol[s];
    const EmitLay L = A.lay[s];
    uint8_t *rd = A.out_reads + A.reads_off[s];
    uint8_t *mf = A.out_maf + A.maf_off[s];
    if (tile == 0) {  // everything of the record that is not a per-base row: once per sub-read
      const RefName N = ref_name(A.S, A.B, r, A.P.glen);
      const uint32_t shown = A.P.sample ? ncol - A.B.nins[s] : wlen;
      const RecLayout LL = rec_layout(A.P, N, read_id, pass, shown, rlen, ncol);
      if (lane == 0) write_headers(A.P, N, LL, rd, mf, read_id, pass, shown, rlen, ncol, minus);
    }
    if (nent == 0) continue;
    const TileGeom g = tile_geom<METHOD>(A, s, r, tile, nent, rlen, ncol, offset, wlen, minus);
    const Ckpt c0 = g.c0;
    const uint32_t e0 = g.e0, e1 = g.e1;
    const bool has_next = g.has_next != 0u;
    const Ckpt *ckp = A.ck + A.B.ck_off[s];
    if (rows_here) {
      uint8_t *seq = rd + L.seq_rel, *qual = rd + L.qual_rel;
      uint8_t *mref = mf + L.refrow_rel, *mread = mf + L.readrow_rel;
      const uint8_t *evbase = A.ev + (A.B.ev_off[s] + (g.segmented ? (uint64_t)tile * PB_SEG_STRIDE : 0ull)) *
                                         (METHOD == PBSIM_METHOD_QSHMM ? 2ull : 1ull);
      RefFetch rf;
      rf.ascii = A.G.ascii;
      rf.offset = offset;
      rf.wlen = wlen;
      rf.minus = minus;
      emit_tile_generic<METHOD, BAM>(evbase, e0, e1, rf, minus, ncol, c0.col, c0.ref, c0.read, seq, qual, mref, mread,
                                     lane, A.philox ? &A.keys : nullptr, (uint32_t)read_id, pass);
    }
    if (A.P.sam) {
      // ip:B:C / pw:B:C arrays: ",9" per read base of this tile (:2324-2331)
      const uint32_t p0 = c0.read;
      const uint32_t p1 = has_next ? ckp[tile + 1].read : rlen;
      uint8_t *ip = rd + L.ip_rel, *pw = rd + L.pw_rel;
      if (BAM) {  // one byte of value 9 per read base
        for (uint32_t j = p0 + lane; j < p1; j += 32u) {
          ip[j] = 9;
          pw[j] = 9;
        }
      } else {
        for (uint32_t j = 2u * p0 + lane; j < 2u * p1; j += 32u) {
          const uint8_t ch = (j & 1u) ? (uint8_t)'9' : (uint8_t)',';
          ip[j] = ch;
          pw[j] = ch;
        }
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------
// K6: statistics of the valid subreads (pbsim.cpp:2293-2316): counters, min/max, the two histograms
// stats block layout (int64): [0] res_num(reads) [1] res_pass_num [2] len_total [3] len_min [4] len_max
//                             [5] sub [6] ins [7] del [8] accuracy sum (2^-40 fixed point) [9..15] spare,
//                             then freq_accuracy[100001], freq_len[...]
// ----------------------------------------------------------------------------------------------
constexpr int kStatCounters = 16;

__global__ void k_stats(Batch B, uint32_t n_sub, uint32_t pass_num, unsigned long long *blk, int64_t freq_len_cells) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long len = 0, nsub = 0, nins = 0, ndel = 0;
  if (s < n_sub) {
    len = B.rlen[s];
    nsub = B.nsub[s];
    nins = B.nins[s];
    ndel = B.ndel[s];
    atomicMin(reinterpret_cast<long long *>(blk + 3), (long long)len);
    atomicMax(reinterpret_cast<long long *>(blk + 4), (long long)len);
    unsigned long long *freq_acc = blk + kStatCounters;
    unsigned long long *freq_len = freq_acc + 100001;
    if ((int64_t)len < freq_len_cells) atomicAdd(&freq_len[len], 1ull);
    // acc_wk = (int)(value * 100000 + 0.5)  (:2315), without FMA contraction
    const double v = __dadd_rn(__dmul_rn(B.accuracy[s], 100000.0), 0.5);
    if (v > -1.0 && v < 100001.0) {
      const int idx = (int)v;
      if (idx >= 0 && idx <= 100000) atomicAdd(&freq_acc[idx], 1ull);
    }
  }
  // warp-aggregate the sums
  for (int o = 16; o > 0; o >>= 1) {
    len += __shfl_down_sync(0xFFFFFFFFu, len, o);
    nsub += __shfl_down_sync(0xFFFFFFFFu, nsub, o);
    nins += __shfl_down_sync(0xFFFFFFFFu, nins, o);
    ndel += __shfl_down_sync(0xFFFFFFFFu, ndel, o);
  }
  // [8]: sum of the per-read accuracies in 2^-40 fixed point — reducible over ranks (pbsim_stats.accuracy_total is
  // the reference's floating-point sum in read order, which is not)
  unsigned long long accfx = 0;
  if (s < n_sub) {
    const double a = B.accuracy[s];
    if (a > 0.0 && a <= 1.0) accfx = (unsigned long long)__double2ll_rn(a * 1099511627776.0);
  }
  for (int o = 16; o > 0; o >>= 1) accfx += __shfl_down_sync(0xFFFFFFFFu, accfx, o);
  if ((threadIdx.x & 31) == 0) {
    if (accfx) atomicAdd(blk + 8, accfx);
    if (len) atomicAdd(blk + 2, len);
    if (nsub) atomicAdd(blk + 5, nsub);
    if (nins) atomicAdd(blk + 6, nins);
    if (ndel) atomicAdd(blk + 7, ndel);
  }
  if (s == 0) {
    atomicAdd(blk + 0, (unsigned long long)(n_sub / pass_num));
    atomicAdd(blk + 1, (unsigned long long)n_sub);
  }
}

}  // namespace pb
