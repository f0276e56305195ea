// Per-read simulation core of the B200 engine: read planning, the qshmm quality chain and the
// errhmm error-state chain, written once for both draw sources (PHILOX / REPLAY).
//
// Pass 1 of the engine: one GPU thread runs the inherently sequential chain of one (read, pass)
// and emits a compact, fixed-rate EVENT STREAM instead of text:
//     qshmm : one uint16 per read position   qv | kind<<7 | info<<9 | ndel<<12
//     errhmm: one uint8  per alignment column kind | info<<2
// plus a checkpoint (column, ref offset, read offset) every PB_TILE entries so that pass 2
// (emit.cuh) can format any tile of any read independently with coalesced loads and stores.
// Reads that touch no non-ACGT base and no bias-relevant homopolymer never look at the genome
// here: substitution / insertion choices are recorded as indices and resolved in pass 2.
//
// Reference behaviour restated (yukiteruono/pbsim3 src/pbsim.cpp):
//     read planning            :2174-2190 (= :3793-3809)
//     qshmm per-position step  :2213-2282
//     errhmm per-column step   :3836-3975
//
// The file compiles as plain C++ as well (tests/hostsim builds it with g++ to check the logic
// against the oracle without a GPU); the product only ever runs it inside CUDA kernels.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define PB_HD __host__ __device__ __forceinline__
#define PB_HD_NOINLINE __host__ __device__ __noinline__
#else
#define PB_HD inline
#define PB_HD_NOINLINE
#endif

#define PB_TILE 1024u        // entries per pass-2 tile / checkpoint interval
#define PB_QS_ROW 100u       // qshmm table resolution
#define PB_ER_ROW 1000u      // errhmm table resolution
#define PB_KIND_MATCH 0u
#define PB_KIND_SUB 1u
#define PB_KIND_INS 2u
#define PB_KIND_DEL 3u       // errhmm column kind; in the qshmm stream kind 3 marks a continuation entry
#define PB_QS_DEL_SAT 15u    // qshmm entry: 15 deletions + "continuation entry follows"
#define PB_QS_CONT_SAT 16383u

namespace pb {

PB_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

PB_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// Philox4x32-10 (Salmon et al., SC'11).  Draw addressing (DESIGN.md):
//   key = (seed, sequence number)   counter = (position, pass << 16, read id, domain)
//   domain 0 planner, 1 the draws of one position, 2 the HMM state draws (one block per 4 positions)
struct Philox {
  uint32_t k0, k1;
  PB_HD void block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) const {
    uint32_t a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint64_t p0 = (uint64_t)0xD2511F53u * c0;  // one IMAD.WIDE gives both halves
      const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
      c0 = (uint32_t)(p1 >> 32) ^ c1 ^ a;
      c1 = (uint32_t)p1;
      c2 = (uint32_t)(p0 >> 32) ^ c3 ^ b;
      c3 = (uint32_t)p0;
      a += 0x9E3779B9u;
      b += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
  }
};

// murmur3 finaliser: a bijection on 32 bits with full avalanche; derives the (rare) second and later
// deletion draws of a position from the Philox word of the first one
PB_HD uint32_t fmix32(uint32_t h) {
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  return h;
}

#define PB_GROUP 4u  // positions whose Philox blocks are computed together (instruction-level parallelism)

// ---------------------------------------------------------------------------------------------
// draw sources.  Purpose-named draws: REPLAY consumes the reference's rand() stream in the
// reference's order (`rand() % m`); PHILOX maps every purpose to a fixed word of the block
// addressed by the position, so results do not depend on scheduling or GPU count.
// ---------------------------------------------------------------------------------------------
struct PhiloxDraw {
  static constexpr bool kCounter = true;  // draws are addressed, not consumed: both branches of a select may be evaluated
  Philox ph;
  uint32_t read_id, pass;
  uint32_t w[4];
  uint32_t g[PB_GROUP][4];
  uint32_t c0w, c1w, c2w, c3w, cidx = 0xFFFFFFFFu;  // chain block (state draws of positions 4*cidx .. 4*cidx+3)
  // state draw of position p: own stream so that the chain can be advanced alone (segment-parallel pass 1)
  PB_HD uint32_t wc(uint32_t p, uint32_t m) {
    if ((p >> 2) != cidx) {
      uint32_t t[4];
      ph.block(p >> 2, pass << 16, read_id, 2u, t);
      c0w = t[0]; c1w = t[1]; c2w = t[2]; c3w = t[3];
      cidx = p >> 2;
    }
    const uint32_t k = p & 3u;
    return mulhi32(k == 0u ? c0w : (k == 1u ? c1w : (k == 2u ? c2w : c3w)), m);
  }
  PB_HD void plan_begin() { ph.block(0u, 0u, read_id, 0u, w); }
  PB_HD uint32_t plan_len(uint32_t m) { return mulhi32(w[0], m); }
  PB_HD uint32_t plan_acc(uint32_t m) { return mulhi32(w[1], m); }
  PB_HD uint32_t plan_off(uint32_t span) { return (uint32_t)mulhi64(((uint64_t)w[2] << 32) | w[3], span); }
  // blocks of positions p .. p+PB_GROUP-1: independent dependency chains the scheduler can interleave
  PB_HD void prefetch(uint32_t p) {
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) ph.block(p + u, pass << 16, read_id, 1u, g[u]);
  }
  PB_HD void begin(uint32_t u) {  // u: index inside the prefetched group (compile-time constant after unrolling)
    w[0] = g[u][0]; w[1] = g[u][1]; w[2] = g[u][2]; w[3] = g[u][3];
  }
  PB_HD uint32_t w0(uint32_t m) { return mulhi32(w[0], m); }
  PB_HD uint32_t w1(uint32_t m) { return mulhi32(w[1], m); }
  PB_HD uint32_t w2(uint32_t m) { return mulhi32(w[2], m); }
  PB_HD uint32_t w3(uint32_t m) { return mulhi32(w[3], m); }
  PB_HD uint32_t choice3() { return ((w[0] & 0xFFFu) * 3u) >> 12; }
  PB_HD uint32_t choice4() { return (w[0] >> 12) & 3u; }
  PB_HD uint32_t choice8() { return w[1] & 7u; }
  PB_HD uint32_t mag3() { return (((w[3] & 0xFFFu) * 3u) >> 12) + 1u; }
  // j-th deletion draw after the current position, on the 0..999999 scale
  PB_HD uint32_t del(uint32_t j) {
    const uint32_t x = (j == 0u) ? w[3] : fmix32(w[3] + j * 0x9E3779B9u);
    return mulhi32(x, 1000000u);
  }
  PB_HD uint32_t consumed() const { return 0; }
};

// PHILOX addressing of the qshmm and sample methods ("v2", DESIGN.md 2.5):
//   error stream   (domain 1): block p >> 1, words 2*(p&1) = X and 2*(p&1)+1 = Y of read position p
//       X: error draw (hit of a threshold t millionths iff X < T32(t)); 3-way choice = ((X & 0xFFF) * 3) >> 12
//       Y: deletion draws (d_0 = Y, d_j = d_{j-1} * 0x9E3779B1 + 0x7F4A7C15); 8-way choice = Y & 7; 4-way choice = (Y >> 3) & 3
//   quality stream (domain 2): block p >> 2, word p & 3 = S
//       state draw = (S >> 16) * modulus >> 16; emission draw = (S & 0xFFFF) * modulus >> 16; freq2qc draw = mulhi(S, modulus)
// T32(t) = min(ceil(t * 2^32 / 10^6), 2^32 - 1): for t < 10^6, X < T32(t) is mulhi32(X, 10^6) < t exactly.
PB_HD uint32_t t32_of(uint32_t t) {
  if (t >= 1000000u) return 0xFFFFFFFFu;
  return (uint32_t)(((uint64_t)t * 4294967296ull + 999999ull) / 1000000ull);
}
// further deletion draws of a position (qshmm / sample): d_0 = Y, d_j = d_{j-1} * 0x9E3779B1 + 0x7F4A7C15
PB_HD uint32_t del_next(uint32_t d) { return d * 0x9E3779B1u + 0x7F4A7C15u; }
#define PB_PROB_SHIFT 26  // PHILOX mode: error probabilities are summed in 2^-26 fixed point (order independent)

struct PhiloxDrawQ {
  static constexpr bool kCounter = true;
  Philox ph;
  uint32_t read_id, pass;
  uint32_t w[4];        // planner block
  uint32_t g[2][4];     // error blocks of the current group of PB_GROUP positions
  uint32_t q[4];        // quality block of the group
  uint32_t X, Y, S;
  PB_HD void plan_begin() { ph.block(0u, 0u, read_id, 0u, w); }
  PB_HD uint32_t plan_len(uint32_t m) { return mulhi32(w[0], m); }
  PB_HD uint32_t plan_acc(uint32_t m) { return mulhi32(w[1], m); }
  PB_HD uint32_t plan_off(uint32_t span) { return (uint32_t)mulhi64(((uint64_t)w[2] << 32) | w[3], span); }
  PB_HD void prefetch(uint32_t p) {  // p is a multiple of PB_GROUP
    ph.block(p >> 1, pass << 16, read_id, 1u, g[0]);
    ph.block((p >> 1) + 1u, pass << 16, read_id, 1u, g[1]);
    ph.block(p >> 2, pass << 16, read_id, 2u, q);
  }
  PB_HD void begin(uint32_t u) {  // u: index inside the group (compile-time constant after unrolling)
    X = g[u >> 1][(u & 1u) * 2u];
    Y = g[u >> 1][(u & 1u) * 2u + 1u];
    S = q[u];
  }
  PB_HD uint32_t qs_state(uint32_t m) { return mulhi32(S & 0xFFFF0000u, m); }
  PB_HD uint32_t qs_emis(uint32_t m) { return mulhi32(S << 16, m); }
  PB_HD uint32_t qs_freq(uint32_t m) { return mulhi32(S, m); }
  PB_HD uint32_t qs_err() { return X; }
  PB_HD uint32_t choice3() { return ((X & 0xFFFu) * 3u) >> 12; }
  PB_HD uint32_t choice4() { return (Y >> 3) & 3u; }
  PB_HD uint32_t choice8() { return Y & 7u; }
  uint32_t dcur;
  PB_HD uint32_t del(uint32_t j) {  // called with j = 0, 1, 2, ... in order
    dcur = (j == 0u) ? Y : del_next(dcur);
    return dcur;
  }
  // a draw against a threshold given on both scales (t6: millionths, t32 = T32(t6))
  static PB_HD bool lt(uint32_t d, uint32_t, uint32_t t32) { return d < t32; }
  PB_HD uint32_t consumed() const { return 0; }
};

struct ReplayDraw {
  static constexpr bool kCounter = false;  // a stream: every draw call consumes one value, in the reference's order
  const int32_t *log;  // the reference's draws
  int64_t cur, end, start;
  PB_HD uint32_t next() {
    const uint32_t v = (cur < end) ? (uint32_t)log[cur] : 0u;
    ++cur;
    return v;
  }
  PB_HD void plan_begin() {}
  PB_HD uint32_t plan_len(uint32_t m) { return next() % m; }
  PB_HD uint32_t plan_acc(uint32_t m) { return next() % m; }
  PB_HD uint32_t plan_off(uint32_t span) { return next() % span; }
  PB_HD void prefetch(uint32_t) {}
  PB_HD void begin(uint32_t) {}
  PB_HD uint32_t wc(uint32_t, uint32_t m) { return next() % m; }
  PB_HD uint32_t w0(uint32_t m) { return next() % m; }
  PB_HD uint32_t w1(uint32_t m) { return next() % m; }
  PB_HD uint32_t w2(uint32_t m) { return next() % m; }
  PB_HD uint32_t w3(uint32_t m) { return next() % m; }
  PB_HD uint32_t choice3() { return next() % 3u; }
  PB_HD uint32_t choice4() { return next() % 4u; }
  PB_HD uint32_t choice8() { return next() % 8u; }
  PB_HD uint32_t mag3() { return next() % 3u + 1u; }
  PB_HD uint32_t del(uint32_t) { return next() % 1000000u; }
  PB_HD uint32_t qs_state(uint32_t m) { return next() % m; }
  PB_HD uint32_t qs_emis(uint32_t m) { return next() % m; }
  PB_HD uint32_t qs_freq(uint32_t m) { return next() % m; }
  PB_HD uint32_t qs_err() { return next() % 1000000u; }
  static PB_HD bool lt(uint32_t d, uint32_t t6, uint32_t) { return d < t6; }
  PB_HD uint32_t consumed() const { return (uint32_t)(cur - start); }
};

// Round keys of Philox4x32-10 for one (seed, sequence): identical for every thread of a launch, so the
// fast path takes them from kernel parameters (constant bank operands) instead of re-deriving them.
struct PhiloxKeys {
  uint32_t k[10][2];
#if !defined(__CUDACC__) || defined(__CUDA_ARCH__) || 1
  PB_HD void init(uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
      k[r][0] = k0 + (uint32_t)r * 0x9E3779B9u;
      k[r][1] = k1 + (uint32_t)r * 0xBB67AE85u;
    }
  }
#endif
};

// (Measured with 7 rounds, the fewest that pass BigCrush: k_sim_seg -10 %, c3 +3.9 %, the latency-bound quality pass
// unchanged.  Not taken: the 10-round generator is the one everybody can check against Random123.)
PB_HD void philox_block_keys(const PhiloxKeys &K, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    c0 = (uint32_t)(p1 >> 32) ^ c1 ^ K.k[r][0];
    c1 = (uint32_t)p1;
    c2 = (uint32_t)(p0 >> 32) ^ c3 ^ K.k[r][1];
    c3 = (uint32_t)p0;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// state-draw words (domain 2) of the PB_GROUP positions starting at p; one block when p is a multiple of 4
PB_HD void chain_words(const PhiloxKeys &K, uint32_t read_id, uint32_t c1, uint32_t p, uint32_t cw[PB_GROUP]) {
  if ((p & 3u) == 0u) {
    philox_block_keys(K, p >> 2, c1, read_id, 2u, cw);
  } else {  // misaligned group (only after a run of >= 15 deletions): two blocks
    uint32_t a[4], b[4];
    philox_block_keys(K, p >> 2, c1, read_id, 2u, a);
    philox_block_keys(K, (p >> 2) + 1u, c1, read_id, 2u, b);
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) {
      const uint32_t q = (p & 3u) + u;  // 1..6
      cw[u] = q == 1u ? a[1] : (q == 2u ? a[2] : (q == 3u ? a[3] : (q == 4u ? b[0] : (q == 5u ? b[1] : b[2]))));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// read planning
// ---------------------------------------------------------------------------------------------
struct PlanTables {
  const int32_t *prob2len;
  const uint8_t *prob2acc;
  uint32_t len_rand_value, acc_rand_value;
  uint32_t len_min;
};

struct ReadPlan {
  uint32_t raw_len;  // prob2len draw before any clipping (the quota test uses it, :2176)
  uint32_t wlen;     // mut.len
  uint32_t offset;   // mut.offset
  uint32_t acc;      // mut.acc
};

// clip_room < 0: no quota clipping (bulk batches); otherwise quota - len_total for this read
template <class Draw>
PB_HD ReadPlan plan_read(const PlanTables &T, Draw &d, uint32_t glen, int64_t clip_room) {
  ReadPlan p;
  d.plan_begin();
  uint32_t len = (uint32_t)T.prob2len[d.plan_len(T.len_rand_value)];
  p.raw_len = len;
  if (clip_room >= 0 && (int64_t)len > clip_room) {
    len = (uint32_t)clip_room;
    if (len < T.len_min) len = T.len_min;
  }
  p.acc = T.prob2acc[d.plan_acc(T.acc_rand_value)];
  if (len >= glen) {
    p.offset = 0;
    len = glen;
  } else {
    p.offset = d.plan_off(glen - len + 1u);
  }
  p.wlen = len;
  return p;
}

// --strategy trans (pbsim.cpp:2842-2866 = :4538-4562): length, accuracy, then the start position from the
// prob2ssp table of the transcript's rank (:2504-2528); the window is clipped at the transcript's end.
// ssp_ends[rank*21 + j]: cumulative table position of start fraction 5*j percent (0xFFFF: row ended), ssp_mod[rank]
// the row modulus.  tlen: length of the transcript.  The returned offset is relative to the transcript.
PB_HD double pb_mul_add_rn(double a, double b, double c) {  // a*b + c with two roundings, as the host computes it
#ifdef __CUDA_ARCH__
  return __dadd_rn(__dmul_rn(a, b), c);
#else
  volatile double m = a * b;
  return m + c;
#endif
}

template <class Draw>
PB_HD ReadPlan plan_read_trans(const PlanTables &T, Draw &d, const uint16_t *ssp_ends, const uint16_t *ssp_mod,
                               uint32_t tlen) {
  ReadPlan p;
  d.plan_begin();
  uint32_t len = (uint32_t)T.prob2len[d.plan_len(T.len_rand_value)];
  p.raw_len = len;
  p.acc = T.prob2acc[d.plan_acc(T.acc_rand_value)];
  const uint32_t rank = (tlen + 999u) / 1000u;  // ceil((double)transcript.len / 1000)
  const uint32_t index = d.plan_off(ssp_mod[rank]) + 1u;
  uint32_t ssp = 100u;
  for (uint32_t j = 0; j < 21u; ++j) {
    const uint32_t e = ssp_ends[rank * 21u + j];
    if (e == 0xFFFFu) break;
    if (index <= e) {
      ssp = j * 5u;
      break;
    }
  }
  const double value = ssp == 0u ? 0.0 : ((double)ssp - 2.5) / 100;
  p.offset = (uint32_t)(int)pb_mul_add_rn((double)tlen, value, 0.5);
  if ((uint64_t)p.offset + len > tlen) len = p.offset < tlen ? tlen - p.offset : 0u;
  p.wlen = len;
  return p;
}

// --strategy templ (:3359-3364 = :5078-5083): one accuracy draw; the read covers the whole template
template <class Draw>
PB_HD ReadPlan plan_read_templ(const PlanTables &T, Draw &d, uint32_t tlen) {
  ReadPlan p;
  d.plan_begin();
  p.acc = T.prob2acc[d.plan_acc(T.acc_rand_value)];
  p.raw_len = tlen;
  p.wlen = tlen;
  p.offset = 0;
  return p;
}

// ---------------------------------------------------------------------------------------------
// slow-path genome access (only reads whose window touches a non-ACGT base or a homopolymer
// with a non-unit deletion bias, or every read when --hp-del-bias != 1)
// ---------------------------------------------------------------------------------------------
struct WindowRef {
  const uint8_t *ascii;   // upper-cased sequence
  const uint8_t *hp4;     // 4-bit homopolymer length per base (low nibble = even index)
  uint32_t offset, wlen;
  uint32_t minus;         // 1: window is the reverse complement
  PB_HD uint32_t gidx(uint32_t r) const { return minus ? offset + wlen - 1u - r : offset + r; }
  PB_HD bool nonacgt(uint32_t r) const {
    const uint8_t c = ascii[gidx(r)];
    return !(c == 'A' || c == 'C' || c == 'G' || c == 'T');
  }
  PB_HD uint32_t hp(uint32_t r) const {
    const uint32_t g = gidx(r);
    return (hp4[g >> 1] >> ((g & 1u) * 4u)) & 15u;
  }
};

struct SubreadResult {
  uint32_t n_entries, rlen, ncol, nsub, nins, ndel;
  uint32_t overflow;
  double accuracy;
};

struct Ckpt {
  uint32_t col, ref, read, pad;
};

// ---------------------------------------------------------------------------------------------
// qshmm
// ---------------------------------------------------------------------------------------------
// Tables of ONE accuracy (staged in shared memory by the kernel).
//   t2[row + k]    : row offset of the next state (= state*100, 16 bit) | transition modulus(next) << 16
//                    | emission modulus(next) << 24 ; row offset 0 is init2state
//   emis[row + k]  : QV
//   freq[k]        : QV when the model has no such accuracy (resolution 1000)
//   thr[qv]        : {sub_thre, ins_thre, max_hp del threshold, del threshold for hp[-1]}
//   thr_hp[qv*12+h]: exact deletion threshold ceil(del_thre[qv] * hp_del_bias[h])
struct QsThr {
  uint32_t sub, ins, del, del0;
};

struct QsFast {  // what the PHILOX fast paths load per quality value
  uint32_t sub, ins, del;  // T32 thresholds: substitution, substitution + insertion, deletion (reference offset > 0)
  uint32_t prob;           // error probability 10^(-qv/10) in 2^-PB_PROB_SHIFT fixed point
};

struct QsView {
  const uint32_t *t2;
  const uint8_t *emis;
  const uint8_t *freq;
  uint32_t has_model, init_mod, freq_mod;
  const QsThr *thr;         // [94]
  const uint32_t *thr_hp;   // [94*12]
  const double *qc_prob;    // [94]
  // PHILOX mode: the same thresholds on the 32-bit scale (T32), and what the position-parallel kernels load
  const QsThr *thr32;       // [94] {T32(sub), T32(ins), T32(del), T32(del0)}
  const uint32_t *thr_hp32; // [94*12]
  const QsFast *fast;       // [94] {T32(sub), T32(ins), T32(del), error probability in 2^-26 fixed point}
};

struct QsSink {
  uint16_t *ev;
  Ckpt *ck;
  uint32_t n, cap;
  uint64_t acc;
  PB_HD void init(uint16_t *e, Ckpt *c, uint32_t capacity) { ev = e; ck = c; n = 0; cap = capacity; acc = 0; }
  PB_HD bool full() const { return n + 2u > cap; }
  PB_HD void checkpoint(uint32_t col, uint32_t ref, uint32_t read) {
    if ((n & (PB_TILE - 1u)) == 0u) {
      Ckpt c; c.col = col; c.ref = ref; c.read = read; c.pad = 0;
      ck[n / PB_TILE] = c;
    }
  }
  PB_HD void push(uint32_t e) {
    acc |= (uint64_t)e << (16u * (n & 3u));
    ++n;
    if ((n & 3u) == 0u) {
      *reinterpret_cast<uint64_t *>(ev + n - 4u) = acc;
      acc = 0;
    }
  }
  PB_HD void flush() {
    const uint32_t rem = n & 3u;
    for (uint32_t i = 0; i < rem; ++i) ev[n - rem + i] = (uint16_t)(acc >> (16u * i));
  }
};

// one position of the qshmm / sample loop after its quality is known: error draw, choices, deletion run.
// Returns the event's kind / info / deletion count; advances R.  Shared by qshmm_simulate and sample_simulate.
template <class Draw, class Bound>
PB_HD void qs_position(const QsView &T, Draw &d, const WindowRef &win, bool slow, uint32_t qv, uint32_t &R,
                       const Bound &more, uint32_t &kind, uint32_t &info, uint32_t &nd) {
  const QsThr th = T.thr[qv];
  QsThr t32 = th;
  if (Draw::kCounter) t32 = T.thr32[qv];
  const uint32_t r = d.qs_err();
  const bool is_sub = Draw::lt(r, th.sub, t32.sub);
  const bool is_ins = !is_sub && Draw::lt(r, th.ins, t32.ins);
  if (Draw::kCounter) {
    info = is_sub ? d.choice3() : (is_ins ? d.choice8() : 0u);
  } else {
    info = 0;
    if (is_sub) info = d.choice3();
    else if (is_ins) info = d.choice8();
  }
  if (slow && is_sub && win.nonacgt(R)) info = d.choice4();  // the %3 draw is still consumed (:2235-2246)
  kind = is_sub ? PB_KIND_SUB : (is_ins ? PB_KIND_INS : PB_KIND_MATCH);
  R += is_ins ? 0u : 1u;
  nd = 0;
  while (more(R)) {
    const uint32_t rd = d.del(nd);
    bool hit = Draw::lt(rd, th.del, t32.del);
    if (hit) {
      if (R == 0u) hit = Draw::lt(rd, th.del0, t32.del0);                                   // mut.hp[-1] (:2269)
      else if (slow) {
        const uint32_t h = qv * 12u + win.hp(R - 1u);
        hit = Draw::lt(rd, T.thr_hp[h], Draw::kCounter ? T.thr_hp32[h] : 0u);
      }
    }
    if (!hit) break;
    ++nd;
    ++R;
  }
}

// the accuracy of a read from its qualities (:2309-2313): the reference's sum in read order (REPLAY), or the
// order-independent fixed-point sum of PHILOX mode
struct QsProbSum {
  double prob = 0.0;
  uint64_t fx = 0;
  template <class Draw>
  PB_HD void add(const QsView &T, uint32_t qv) {
    if (Draw::kCounter) fx += T.fast[qv].prob;
    else prob += T.qc_prob[qv];
  }
  template <class Draw>
  PB_HD double accuracy(uint32_t P) const {
    const double p = Draw::kCounter ? (double)fx / (double)(1u << PB_PROB_SHIFT) : prob;
    return 1.0 - (p / (double)P);
  }
};

template <class Draw>
PB_HD void qshmm_simulate(const QsView &T, Draw &d, const WindowRef &win, bool slow, uint32_t wlen,
                          QsSink &sink, SubreadResult &res) {
  uint32_t R = 0, P = 0, C = 0;
  uint32_t row = 0, mod = T.init_mod, emod = 1;
  uint32_t nsub = 0, nins = 0, ndel = 0;
  QsProbSum ps;
  res.overflow = 0;
  const auto more = [wlen](uint32_t r) { return r < wlen; };
  while (R < wlen) {
    d.prefetch(P);
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) {
      if (R >= wlen) break;
      if (sink.full()) { res.overflow = 1; break; }
      sink.checkpoint(C, R, P);
      d.begin(u);
      uint32_t qv;
      if (T.has_model) {
        const uint32_t t = T.t2[row + d.qs_state(mod)];
        row = t & 0xFFFFu;
        mod = (t >> 16) & 0xFFu;
        emod = t >> 24;
        qv = T.emis[row + d.qs_emis(emod)];
      } else {
        qv = T.freq[d.qs_freq(T.freq_mod)];
      }
      ps.template add<Draw>(T, qv);
      uint32_t kind, info, nd;
      qs_position(T, d, win, slow, qv, R, more, kind, info, nd);
      nsub += kind == PB_KIND_SUB ? 1u : 0u;
      nins += kind == PB_KIND_INS ? 1u : 0u;
      ++P;
      ++C;
      ndel += nd;
      C += nd;
      const uint32_t base = qv | (kind << 7) | (info << 9);
      if (nd < PB_QS_DEL_SAT) {
        sink.push(base | (nd << 12));
      } else {
        sink.push(base | (PB_QS_DEL_SAT << 12));
        uint32_t rest = nd - PB_QS_DEL_SAT;
        for (;;) {  // continuation entries: 14-bit counts, 16383 = "more follows"
          if (sink.full()) { res.overflow = 1; break; }
          sink.checkpoint(C - rest, R - rest, P);  // a tile may start here: state before these deletions
          const uint32_t c = rest < PB_QS_CONT_SAT ? rest : PB_QS_CONT_SAT;
          sink.push((c & 0x7Fu) | (3u << 7) | ((c >> 7) << 9));
          if (c < PB_QS_CONT_SAT) break;
          rest -= PB_QS_CONT_SAT;
        }
        if (res.overflow) break;
      }
    }
    if (res.overflow) break;
  }
  sink.flush();
  res.n_entries = sink.n;
  res.rlen = P;
  res.ncol = C;
  res.nsub = nsub;
  res.nins = nins;
  res.ndel = ndel;
  res.accuracy = ps.template accuracy<Draw>(P);  // :2313 (accuracy from the emitted qualities)
}

// ---------------------------------------------------------------------------------------------
// --method sample (simulate_by_sample, pbsim.cpp:1775-1833): the quality string of a sampled read gives
// the quality of every position, so there is no chain; the per-position draws and the event stream are
// those of qshmm.  `len` (mut.len, :1756-1763) bounds BOTH the window and the read, and no deletion is
// drawn once either is used up.  The read's accuracy sums the error probabilities in read order (:1868).
// ---------------------------------------------------------------------------------------------
template <class Draw>
PB_HD void sample_simulate(const QsView &T, Draw &d, const WindowRef &win, bool slow, uint32_t len,
                           const uint8_t *quals, QsSink &sink, SubreadResult &res) {
  uint32_t R = 0, P = 0, C = 0;
  uint32_t nsub = 0, nins = 0, ndel = 0;
  QsProbSum ps;
  res.overflow = 0;
  while (R < len && P < len) {
    d.prefetch(P);
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) {
      if (R >= len || P >= len) break;
      if (sink.full()) { res.overflow = 1; break; }
      sink.checkpoint(C, R, P);
      d.begin(u);
      const uint32_t qv = (uint32_t)quals[P] - 33u;
      ps.template add<Draw>(T, qv);
      ++P;
      const uint32_t Pn = P;
      const auto more = [len, Pn](uint32_t r) { return r < len && Pn < len; };
      uint32_t kind, info, nd;
      qs_position(T, d, win, slow, qv, R, more, kind, info, nd);
      nsub += kind == PB_KIND_SUB ? 1u : 0u;
      nins += kind == PB_KIND_INS ? 1u : 0u;
      ++C;
      ndel += nd;
      C += nd;
      const uint32_t base = qv | (kind << 7) | (info << 9);
      if (nd < PB_QS_DEL_SAT) {
        sink.push(base | (nd << 12));
      } else {
        sink.push(base | (PB_QS_DEL_SAT << 12));
        uint32_t rest = nd - PB_QS_DEL_SAT;
        for (;;) {
          if (sink.full()) { res.overflow = 1; break; }
          sink.checkpoint(C - rest, R - rest, P);
          const uint32_t c = rest < PB_QS_CONT_SAT ? rest : PB_QS_CONT_SAT;
          sink.push((c & 0x7Fu) | (3u << 7) | ((c >> 7) << 9));
          if (c < PB_QS_CONT_SAT) break;
          rest -= PB_QS_CONT_SAT;
        }
        if (res.overflow) break;
      }
    }
    if (res.overflow) break;
  }
  sink.flush();
  res.n_entries = sink.n;
  res.rlen = P;
  res.ncol = C;
  res.nsub = nsub;
  res.nins = nins;
  res.ndel = ndel;
  res.accuracy = ps.template accuracy<Draw>(P);
}

// ---------------------------------------------------------------------------------------------
// qshmm fast path: PHILOX draws, reads that never need the genome in pass 1 (not `slow`).
// Same results as qshmm_simulate<PhiloxDrawQ> entry for entry, except that the stream is padded with
// no-op entries (continuation entries with count 0) to a multiple of PB_GROUP, which lets every group of
// 4 positions be packed in registers and written with one 8-byte store, checks run once per group and the
// common path stay free of divergent branches.
// ---------------------------------------------------------------------------------------------
#define PB_QS_PAD (3u << 7)  // continuation entry, count 0

// error-stream words of the PB_GROUP positions starting at p (a multiple of 4): x[u], y[u]
PB_HD void error_words(const PhiloxKeys &K, uint32_t read_id, uint32_t c1, uint32_t p, uint32_t x[PB_GROUP], uint32_t y[PB_GROUP]) {
  uint32_t a[4], b[4];
  philox_block_keys(K, p >> 1, c1, read_id, 1u, a);
  philox_block_keys(K, (p >> 1) + 1u, c1, read_id, 1u, b);
  x[0] = a[0]; y[0] = a[1]; x[1] = a[2]; y[1] = a[3];
  x[2] = b[0]; y[2] = b[1]; x[3] = b[2]; y[3] = b[3];
}
// the words of ONE position (any p): used off the hot paths
PB_HD void error_words_at(const PhiloxKeys &K, uint32_t read_id, uint32_t c1, uint32_t p, uint32_t &x, uint32_t &y) {
  uint32_t a[4];
  philox_block_keys(K, p >> 1, c1, read_id, 1u, a);
  x = (p & 1u) ? a[2] : a[0];
  y = (p & 1u) ? a[3] : a[1];
}

// kind, info and deletion count of one position from its quality and its two error-stream words, for a position
// whose reference offset is > 0 after the base (every position except leading insertions of a read).
// The first two deletion draws are evaluated without a branch (the second is one multiply-add away from the first).
PB_HD uint32_t qs_event(const QsFast th, uint32_t qv, uint32_t X, uint32_t Y, uint32_t &nd) {
  const bool is_sub = X < th.sub;
  const bool is_ins = !is_sub && X < th.ins;  // (the insertion threshold is cumulative)
  const uint32_t c3 = mulhi32(X << 20, 3u);    // ((X & 0xFFF) * 3) >> 12
  uint32_t e = qv;
  if (is_sub) e |= (PB_KIND_SUB << 7) | (c3 << 9);
  if (is_ins) e |= (PB_KIND_INS << 7) | ((Y & 7u) << 9);
  const uint32_t y2 = del_next(Y);
  const bool hit1 = Y < th.del, hit2 = hit1 && y2 < th.del;
  nd = (hit1 ? 1u : 0u) + (hit2 ? 1u : 0u);
  if (hit2) {
    uint32_t d = y2;
    while (nd < (1u << 20)) {
      d = del_next(d);
      if (!(d < th.del)) break;
      ++nd;
    }
  }
  return e;
}

PB_HD void qshmm_simulate_fast(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass,
                               uint32_t wlen, uint16_t *ev, Ckpt *ck, uint32_t cap, SubreadResult &res) {
  uint32_t R = 0, P = 0, n = 0;
  uint32_t row = 0, mod = T.init_mod, emod = 1;
  uint32_t nsub = 0, ndel = 0;
  uint64_t prob = 0;
  res.overflow = 0;
  const uint32_t c1 = pass << 16;
  while (R < wlen) {
    if (n + 2u * PB_GROUP > cap) { res.overflow = 1; break; }
    if ((n & (PB_TILE - 1u)) == 0u) {
      Ckpt c; c.col = P + ndel; c.ref = R; c.read = P; c.pad = 0;
      ck[n / PB_TILE] = c;
    }
    // P is a multiple of PB_GROUP here: a group is only cut short by the end of the read
    uint32_t x[PB_GROUP], y[PB_GROUP], q[PB_GROUP];
    error_words(K, read_id, c1, P, x, y);
    philox_block_keys(K, P >> 2, c1, read_id, 2u, q);
    uint32_t e[PB_GROUP];
    uint32_t big_u = PB_GROUP, big_nd = 0;  // rare: an entry with >= 15 deletions ends the group early
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) {
      e[u] = PB_QS_PAD;
      if (R < wlen && big_u == PB_GROUP) {
        uint32_t qv;
        if (T.has_model) {
          const uint32_t t = T.t2[row + mulhi32(q[u] & 0xFFFF0000u, mod)];
          row = t & 0xFFFFu;
          mod = (t >> 16) & 0xFFu;
          emod = t >> 24;
          qv = T.emis[row + mulhi32(q[u] << 16, emod)];
        } else {
          qv = T.freq[mulhi32(q[u], T.freq_mod)];
        }
        const QsFast th = T.fast[qv];
        prob += th.prob;
        const bool is_sub = x[u] < th.sub;
        const bool is_err = x[u] < th.ins;
        const uint32_t c3 = ((x[u] & 0xFFFu) * 3u) >> 12, c8 = y[u] & 7u;
        const uint32_t info = is_sub ? c3 : (is_err ? c8 : 0u);
        const uint32_t kind = is_sub ? PB_KIND_SUB : (is_err ? PB_KIND_INS : PB_KIND_MATCH);
        nsub += is_sub ? 1u : 0u;
        R += (is_err && !is_sub) ? 0u : 1u;
        ++P;
        uint32_t nd = 0;
        if (R < wlen && y[u] < (R != 0u ? th.del : T.thr32[qv].del0)) {
          nd = 1;
          ++R;
          for (uint32_t d = del_next(y[u]); R < wlen && d < th.del; d = del_next(d)) {
            ++nd;
            ++R;
          }
        }
        ndel += nd;
        const uint32_t base = qv | (kind << 7) | (info << 9);
        if (nd < PB_QS_DEL_SAT) {
          e[u] = base | (nd << 12);
        } else {
          e[u] = base | (PB_QS_DEL_SAT << 12);
          big_u = u;
          big_nd = nd - PB_QS_DEL_SAT;
        }
      }
    }
    uint64_t *dst = reinterpret_cast<uint64_t *>(ev + n);
    *dst = (uint64_t)(e[0] | (e[1] << 16)) | ((uint64_t)(e[2] | (e[3] << 16)) << 32);
    n += PB_GROUP;
    if (big_u != PB_GROUP) {
      // continuation entries directly follow their entry, then the rest of the group follows them: the group's
      // remaining positions are redone one entry at a time so that P stays a multiple of PB_GROUP afterwards
      n -= PB_GROUP - 1u - big_u;          // drop the entries after the big one
      uint32_t rest = big_nd;
      for (;;) {
        if (n + 2u * PB_GROUP > cap) { res.overflow = 1; break; }
        if ((n & (PB_TILE - 1u)) == 0u) {  // a tile may start here: state before these deletions
          Ckpt c; c.col = P + ndel - rest; c.ref = R - rest; c.read = P; c.pad = 0;
          ck[n / PB_TILE] = c;
        }
        const uint32_t c = rest < PB_QS_CONT_SAT ? rest : PB_QS_CONT_SAT;
        ev[n++] = (uint16_t)((c & 0x7Fu) | (3u << 7) | ((c >> 7) << 9));
        if (c < PB_QS_CONT_SAT) break;
        rest -= PB_QS_CONT_SAT;
      }
      if (res.overflow) break;
      // the positions of the group behind the big entry, each followed by its own continuation entries
      for (uint32_t u = big_u + 1u; u < PB_GROUP && R < wlen; ++u) {
        if (n + 2u * PB_GROUP > cap) { res.overflow = 1; break; }
        if ((n & (PB_TILE - 1u)) == 0u) {
          Ckpt c; c.col = P + ndel; c.ref = R; c.read = P; c.pad = 0;
          ck[n / PB_TILE] = c;
        }
        uint32_t qv;
        if (T.has_model) {
          const uint32_t t = T.t2[row + mulhi32(q[u] & 0xFFFF0000u, mod)];
          row = t & 0xFFFFu;
          mod = (t >> 16) & 0xFFu;
          emod = t >> 24;
          qv = T.emis[row + mulhi32(q[u] << 16, emod)];
        } else {
          qv = T.freq[mulhi32(q[u], T.freq_mod)];
        }
        const QsFast th = T.fast[qv];
        prob += th.prob;
        const bool is_sub = x[u] < th.sub;
        const bool is_err = x[u] < th.ins;
        const uint32_t info = is_sub ? (((x[u] & 0xFFFu) * 3u) >> 12) : (is_err ? (y[u] & 7u) : 0u);
        const uint32_t kind = is_sub ? PB_KIND_SUB : (is_err ? PB_KIND_INS : PB_KIND_MATCH);
        nsub += is_sub ? 1u : 0u;
        R += (is_err && !is_sub) ? 0u : 1u;
        ++P;
        uint32_t nd = 0;
        if (R < wlen && y[u] < (R != 0u ? th.del : T.thr32[qv].del0)) {
          nd = 1;
          ++R;
          for (uint32_t d = del_next(y[u]); R < wlen && d < th.del; d = del_next(d)) { ++nd; ++R; }
        }
        ndel += nd;
        const uint32_t base = qv | (kind << 7) | (info << 9);
        ev[n++] = (uint16_t)(base | ((nd < PB_QS_DEL_SAT ? nd : PB_QS_DEL_SAT) << 12));
        uint32_t rest2 = nd >= PB_QS_DEL_SAT ? nd - PB_QS_DEL_SAT : 0u;
        bool cont = nd >= PB_QS_DEL_SAT;
        while (cont) {
          if (n + 2u * PB_GROUP > cap) { res.overflow = 1; break; }
          if ((n & (PB_TILE - 1u)) == 0u) {
            Ckpt c; c.col = P + ndel - rest2; c.ref = R - rest2; c.read = P; c.pad = 0;
            ck[n / PB_TILE] = c;
          }
          const uint32_t c = rest2 < PB_QS_CONT_SAT ? rest2 : PB_QS_CONT_SAT;
          ev[n++] = (uint16_t)((c & 0x7Fu) | (3u << 7) | ((c >> 7) << 9));
          cont = c >= PB_QS_CONT_SAT;
          rest2 -= c;
        }
        if (res.overflow) break;
      }
      if (res.overflow) break;
      while (n & (PB_GROUP - 1u)) {         // re-align; a checkpoint can only fall on a group boundary
        ev[n++] = (uint16_t)PB_QS_PAD;
      }
    }
  }
  res.n_entries = n;
  res.rlen = P;
  res.ncol = P + ndel;
  res.nsub = nsub;
  res.ndel = ndel;
  res.nins = P + ndel - R;  // C = P + ndel and R = P - nins + ndel
  res.accuracy = 1.0 - (((double)prob / (double)(1u << PB_PROB_SHIFT)) / (double)P);
}

// ---------------------------------------------------------------------------------------------
// qshmm SEGMENT-PARALLEL pass 1 (PHILOX, reads that never need the genome in pass 1).
// A read is cut into segments of PB_TILE read positions; the work is split by what is sequential and what is not:
//   * the QUALITY pass: the HMM chain is the only sequential part of a read.  One thread walks a chunk of segments
//     through the chain (its own Philox stream, one block per 4 positions).  The state entering a chunk is
//     recovered EXACTLY by backward coupling: run every reachable state through the positions just before the
//     chunk with those positions' own draws; as soon as all images coincide the state is independent of the
//     earlier history (if the window reaches position 0 the init draw decides).
//   * the ERROR pass: given its quality, a position depends on nothing but its own two error-stream words: error
//     draw, choices, deletion run -> the event.
//   Model accuracies run both in the same thread (k_qs_pass1, qshmm_chunk_pass1): the chain's lookups leave issue
//   slots free that the error pass's arithmetic fills, and a quality never travels through memory.  Accuracies
//   without a model have no chain: one WARP handles a segment (k_sim_seg), consecutive lanes on consecutive
//   positions, qualities from the freq2qc table.
// Segments are simulated "unbounded" (they cannot know the reference offset they start at); find_end then locates
// the position at which the window is used up, clips the last deletion run and drops the rest, which is what the
// sequential loop `while (ref_offset < mut.len)` (:2213, :2268) does.
// ---------------------------------------------------------------------------------------------
#define PB_SEG_SLACK 64u                       // extra entries per segment slot (continuation entries, pads)
#define PB_SEG_STRIDE (PB_TILE + PB_SEG_SLACK) // entries between consecutive segment slots of a read

struct QsSegAux {            // per accuracy, beside the QsView tables
  const uint8_t *tmod;       // [51] transition modulus of a state
  const uint8_t *emodv;      // [51] emission modulus of a state
  uint64_t reach;            // states reachable from the init distribution (bit s)
};

struct SegResult {
  uint32_t n_entries, ref_adv, nsub, ndel;
  uint32_t flags;            // 1: slot overflow, 2: coupling window exhausted
  uint32_t pad;
  uint64_t prob;             // qshmm: fixed-point sum of the error probabilities; errhmm: the insertion count
};

PB_HD uint32_t qs_state_of_row(uint32_t row) { return (row * 41944u) >> 22; }  // row / 100 for row <= 5100

// state entering position p_start (>= 1).  The window doubles until all images coalesce; when it reaches
// position 0 the init draw decides, so the search always ends with the exact state.
PB_HD bool qshmm_segment_start(const QsView &T, const QsSegAux &A, const PhiloxKeys &K, uint32_t read_id,
                               uint32_t pass, uint32_t p_start, uint32_t first_window, uint32_t &row, uint32_t &mod,
                               uint32_t &emod) {
  const uint32_t c1 = pass << 16;
  for (uint32_t B = first_window;; B *= 2u) {
    const bool from_zero = p_start <= B;
    const uint32_t p0 = from_zero ? 0u : p_start - B;
    uint64_t mask = from_zero ? 1ull : A.reach;  // from position 0: the virtual state 0 (row 0 = init2state)
    uint32_t s_row = 0, s_mod = T.init_mod, s_emod = 1;
    bool single = from_zero;
    uint32_t cwb[4] = {0, 0, 0, 0};
    for (uint32_t p = p0; p < p_start; ++p) {
      if (p == p0 || (p & 3u) == 0u) philox_block_keys(K, p >> 2, c1, read_id, 2u, cwb);
      const uint32_t k4 = p & 3u;
      const uint32_t wdraw = (k4 == 0u ? cwb[0] : (k4 == 1u ? cwb[1] : (k4 == 2u ? cwb[2] : cwb[3]))) & 0xFFFF0000u;
      if (single) {
        const uint32_t t = T.t2[s_row + mulhi32(wdraw, s_mod)];
        s_row = t & 0xFFFFu;
        s_mod = (t >> 16) & 0xFFu;
        s_emod = t >> 24;
      } else {
        uint64_t next = 0;
        uint32_t last_t = 0;
        for (uint64_t m = mask; m; m &= m - 1ull) {
#if defined(__CUDA_ARCH__)
          const uint32_t s = (uint32_t)__ffsll((long long)m) - 1u;
#else
          const uint32_t s = (uint32_t)__builtin_ctzll(m);
#endif
          last_t = T.t2[s * PB_QS_ROW + mulhi32(wdraw, A.tmod[s])];
          next |= 1ull << qs_state_of_row(last_t & 0xFFFFu);
        }
        mask = next;
        if ((mask & (mask - 1ull)) == 0ull) {  // coalesced: one image left
          single = true;
          s_row = last_t & 0xFFFFu;
          s_mod = (last_t >> 16) & 0xFFu;
          s_emod = last_t >> 24;
        }
      }
    }
    if (single) {
      row = s_row; mod = s_mod; emod = s_emod;
      return true;
    }
  }
}

PB_HD void store_u16x8(uint16_t *dst, const uint32_t v[4]) {  // dst is 16-byte aligned
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<uint4 *>(dst) = make_uint4(v[0], v[1], v[2], v[3]);
#else
  for (int i = 0; i < 4; ++i) { dst[2 * i] = (uint16_t)v[i]; dst[2 * i + 1] = (uint16_t)(v[i] >> 16); }
#endif
}

// QUALITY pass alone over segments k_from .. k_to-1 of a read from the state (row, mod, emod) that enters segment
// k_from: the quality value of every position goes into bits 0-6 of its entry in the segment's slot, for
// qshmm_error_segment to turn into events.  The kernels run both passes in one walk (qshmm_chunk_pass1); this split
// statement is what the CPU harness runs, and the reference the fused walk is tested against.
PB_HD void qshmm_quality_range(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass, uint32_t row,
                               uint32_t mod, uint32_t emod, uint32_t k_from, uint32_t k_to, uint16_t *slots) {
  const uint32_t c1 = pass << 16;
  uint32_t nx[8];
  philox_block_keys(K, (k_from * PB_TILE) >> 2, c1, read_id, 2u, nx);
  philox_block_keys(K, ((k_from * PB_TILE) >> 2) + 1u, c1, read_id, 2u, nx + 4);
  for (uint32_t k = k_from; k < k_to; ++k) {
    uint16_t *slot = slots + (uint64_t)k * PB_SEG_STRIDE;
    for (uint32_t j = 0; j < PB_TILE; j += 8u) {
      const uint32_t p = k * PB_TILE + j;
      uint32_t cw[8];
#pragma unroll
      for (uint32_t u = 0; u < 8u; ++u) cw[u] = nx[u];
      philox_block_keys(K, (p >> 2) + 2u, c1, read_id, 2u, nx);
      philox_block_keys(K, (p >> 2) + 3u, c1, read_id, 2u, nx + 4);
      uint32_t out[4];
#pragma unroll
      for (uint32_t u = 0; u < 8u; ++u) {
        const uint32_t t = T.t2[row + mulhi32(cw[u] & 0xFFFF0000u, mod)];
        row = t & 0xFFFFu;
        mod = (t >> 16) & 0xFFu;
        emod = t >> 24;
        const uint32_t qv = T.emis[row + mulhi32(cw[u] << 16, emod)];
        if (u & 1u) out[u >> 1] |= qv << 16;
        else out[u >> 1] = qv;
      }
      store_u16x8(slot + j, out);
    }
  }
}

// the qualities of PB_GROUP positions of an accuracy WITHOUT model (freq2qc table, :2230): no chain, so the
// error pass computes them itself
PB_HD void qs_freq_qualities(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t c1, uint32_t p,
                             uint32_t qv[PB_GROUP]) {
  uint32_t q[4];
  philox_block_keys(K, p >> 2, c1, read_id, 2u, q);
#pragma unroll
  for (uint32_t u = 0; u < PB_GROUP; ++u) qv[u] = T.freq[mulhi32(q[u], T.freq_mod)];
}

// ERROR pass, the work of one lane: the events of positions p .. p+3 (p a multiple of 4) from their qualities,
// packed two per word (w0: positions p, p+1; w1: p+2, p+3).  Deletion counts are stored saturated at
// PB_QS_DEL_SAT; `big` reports that one of them was (the segment is then redone by qshmm_segment_generic, which
// writes continuation entries).  The counters are taken from the packed events (sub: bit 7, ins: bit 8, deletions:
// bits 12-15 of every half word).
struct QsLaneTotals {
  uint32_t nsub, nins, ndel, prob, big;
};
PB_HD uint32_t pb_popc(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__popc(x);
#else
  return (uint32_t)__builtin_popcount(x);
#endif
}
// qs_error_group: the same from the positions' error-stream words (error_words) given; qs_error_lane computes them
PB_HD void qs_error_group(const QsFast *fast, const uint32_t qv[PB_GROUP], const uint32_t x[PB_GROUP],
                          const uint32_t y[PB_GROUP], uint32_t &w0, uint32_t &w1, QsLaneTotals &t) {
  uint32_t e[PB_GROUP];
#pragma unroll
  for (uint32_t u = 0; u < PB_GROUP; ++u) {
    const QsFast th = fast[qv[u]];
    uint32_t nd;
    const uint32_t base = qs_event(th, qv[u], x[u], y[u], nd);
    t.prob += th.prob;
    t.big |= nd >= PB_QS_DEL_SAT ? 1u : 0u;
    e[u] = base | ((nd < PB_QS_DEL_SAT ? nd : PB_QS_DEL_SAT) << 12);
  }
  w0 = e[0] | (e[1] << 16);
  w1 = e[2] | (e[3] << 16);
  t.nsub += pb_popc((w0 & 0x00800080u) | ((w1 & 0x00800080u) << 1));
  t.nins += pb_popc((w0 & 0x01000100u) | ((w1 & 0x01000100u) << 1));
  const uint32_t dd = ((w0 >> 12) & 0x000F000Fu) + ((w1 >> 12) & 0x000F000Fu);
  t.ndel += (dd & 0xFFFFu) + (dd >> 16);
}
PB_HD void qs_error_lane(const QsFast *fast, const PhiloxKeys &K, uint32_t read_id, uint32_t c1, uint32_t p,
                         const uint32_t qv[PB_GROUP], uint32_t &w0, uint32_t &w1, QsLaneTotals &t) {
  uint32_t x[PB_GROUP], y[PB_GROUP];
  error_words(K, read_id, c1, p, x, y);
  qs_error_group(fast, qv, x, y, w0, w1, t);
}

// ERROR pass, first segment of a read: while the reference offset is still 0 (leading insertions) the deletion
// test uses the threshold of mut.hp[-1] (:2269) instead of the one qs_event applied.  Walks the leading
// insertions of the slot, corrects their deletion counts and returns the deletions removed.
PB_HD uint32_t qs_fix_leading(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t c1, uint16_t *ev) {
  uint32_t removed = 0;
  for (uint32_t p = 0; p < PB_TILE; ++p) {
    const uint32_t v = ev[p];
    if (((v >> 7) & 3u) != PB_KIND_INS) break;     // a base that consumes the reference: offset > 0 from here on
    uint32_t x, y;
    error_words_at(K, read_id, c1, p, x, y);
    if (y < T.thr32[v & 0x7Fu].del0) break;        // deleted under the hp[-1] rule as well (del0 <= del): unchanged
    removed += v >> 12;
    ev[p] = (uint16_t)(v & 0x0FFFu);
  }
  return removed;
}

// ERROR pass, generic statement for one whole segment: entries with >= PB_QS_DEL_SAT deletions get continuation
// entries, the hp[-1] rule is applied as the positions go.  qv: the qualities of the segment's PB_TILE positions
// (model accuracies; ignored otherwise).  Used for the rare segments qs_error_lane reports as `big`.
PB_HD void qshmm_segment_generic(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass,
                                 uint32_t p_start, bool first_segment, const uint8_t *qv_in, uint16_t *ev,
                                 SegResult &res) {
  uint32_t R = first_segment ? 0u : 1u;  // only "is it still 0" matters; ref_adv is counted separately
  uint32_t radv = 0, n = 0, nsub = 0, ndel = 0;
  uint64_t prob = 0;
  const uint32_t c1 = pass << 16;
  res.flags = 0;
  for (uint32_t j = 0; j < PB_TILE; ++j) {
    if (n + 2u * PB_GROUP > PB_SEG_STRIDE) { res.flags |= 1u; break; }
    const uint32_t P = p_start + j;
    uint32_t qv;
    if (T.has_model) {
      qv = qv_in[j];
    } else {
      uint32_t q[4];
      philox_block_keys(K, P >> 2, c1, read_id, 2u, q);
      const uint32_t k4 = P & 3u;
      qv = T.freq[mulhi32(k4 == 0u ? q[0] : (k4 == 1u ? q[1] : (k4 == 2u ? q[2] : q[3])), T.freq_mod)];
    }
    uint32_t x, y;
    error_words_at(K, read_id, c1, P, x, y);
    const QsFast th = T.fast[qv];
    prob += th.prob;
    const bool is_sub = x < th.sub;
    const bool is_err = x < th.ins;
    const uint32_t info = is_sub ? (((x & 0xFFFu) * 3u) >> 12) : (is_err ? (y & 7u) : 0u);
    const uint32_t kind = is_sub ? PB_KIND_SUB : (is_err ? PB_KIND_INS : PB_KIND_MATCH);
    nsub += is_sub ? 1u : 0u;
    const uint32_t a = (is_err && !is_sub) ? 0u : 1u;
    R += a;
    radv += a;
    uint32_t nd = 0;
    if (y < (R != 0u ? th.del : T.thr32[qv].del0)) {
      nd = 1;
      for (uint32_t d = del_next(y); nd < (1u << 20) && d < th.del; d = del_next(d)) ++nd;
      R += nd;
      radv += nd;
    }
    ndel += nd;
    const uint32_t base = qv | (kind << 7) | (info << 9);
    if (nd < PB_QS_DEL_SAT) {
      ev[n++] = (uint16_t)(base | (nd << 12));
    } else {
      ev[n++] = (uint16_t)(base | (PB_QS_DEL_SAT << 12));
      uint32_t rest = nd - PB_QS_DEL_SAT;
      for (;;) {
        if (n + 2u * PB_GROUP > PB_SEG_STRIDE) { res.flags |= 1u; break; }
        const uint32_t c = rest < PB_QS_CONT_SAT ? rest : PB_QS_CONT_SAT;
        ev[n++] = (uint16_t)((c & 0x7Fu) | (3u << 7) | ((c >> 7) << 9));
        if (c < PB_QS_CONT_SAT) break;
        rest -= PB_QS_CONT_SAT;
      }
      if (res.flags) break;
    }
  }
  while (n & (PB_GROUP - 1u)) ev[n++] = (uint16_t)PB_QS_PAD;
  res.n_entries = n;
  res.ref_adv = radv;
  res.nsub = nsub;
  res.ndel = ndel;
  res.pad = 0;
  res.prob = prob;
}

// ERROR pass over one segment, as the warp of k_sim_seg runs it (sequential statement for the CPU harness: the
// 256 lane steps one after the other).  With T.has_model the slot holds the qualities on entry (qshmm_quality_range's,
// or --method sample: the pool entry's); otherwise they come from the freq2qc table.
PB_HD void qshmm_error_segment(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass, uint32_t p_start,
                               bool first_segment, uint16_t *ev, SegResult &res) {
  const uint32_t c1 = pass << 16;
  QsLaneTotals t;
  t.nsub = t.nins = t.ndel = t.prob = t.big = 0;
  uint64_t prob = 0;
  uint8_t qsave[PB_TILE];
  for (uint32_t j = 0; j < PB_TILE; j += PB_GROUP) {
    uint32_t qv[PB_GROUP], e[PB_GROUP];
    if (T.has_model) {
#pragma unroll
      for (uint32_t u = 0; u < PB_GROUP; ++u) qv[u] = ev[j + u] & 0x7Fu;
    } else {
      qs_freq_qualities(T, K, read_id, c1, p_start + j, qv);
    }
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) qsave[j + u] = (uint8_t)qv[u];
    t.prob = 0;
    uint32_t w0, w1;
    qs_error_lane(T.fast, K, read_id, c1, p_start + j, qv, w0, w1, t);
    e[0] = w0 & 0xFFFFu; e[1] = w0 >> 16; e[2] = w1 & 0xFFFFu; e[3] = w1 >> 16;
    prob += t.prob;
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) ev[j + u] = (uint16_t)e[u];
  }
  if (t.big) {
    qshmm_segment_generic(T, K, read_id, pass, p_start, first_segment, qsave, ev, res);
    return;
  }
  if (first_segment) t.ndel -= qs_fix_leading(T, K, read_id, c1, ev);
  res.n_entries = PB_TILE;
  res.ref_adv = PB_TILE - t.nins + t.ndel;
  res.nsub = t.nsub;
  res.ndel = t.ndel;
  res.flags = 0;
  res.pad = 0;
  res.prob = prob;
}

// PASS 1 of segments k_from .. k_to-1 of a read of a MODEL accuracy, from the state (row, mod) that enters segment
// k_from: the quality pass (chain + emission lookups) and the error pass (qs_error_group) of every position in one
// walk, 8 positions per group, whose events go out with one 16-byte store; the totals of segment k go to res[k].
// The lookups form one dependent chain (table entry -> next row); the Philox blocks of a group (chain words of the
// NEXT group, error words of this one) do not depend on it and are computed alongside.  A quality is never stored on
// its own: a segment with an entry of >= PB_QS_DEL_SAT deletions (rare) takes its qualities back from bits 0-6 of the
// events it wrote and is redone by qshmm_segment_generic.
PB_HD void qshmm_chunk_pass1(const QsView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass, uint32_t row,
                             uint32_t mod, uint32_t k_from, uint32_t k_to, uint16_t *slots, SegResult *res) {
  const uint32_t c1 = pass << 16;
  uint32_t nx[8];
  philox_block_keys(K, (k_from * PB_TILE) >> 2, c1, read_id, 2u, nx);
  philox_block_keys(K, ((k_from * PB_TILE) >> 2) + 1u, c1, read_id, 2u, nx + 4);
  for (uint32_t k = k_from; k < k_to; ++k) {
    uint16_t *slot = slots + (uint64_t)k * PB_SEG_STRIDE;
    QsLaneTotals t;
    t.nsub = t.nins = t.ndel = t.prob = t.big = 0;
    uint64_t prob = 0;
    for (uint32_t j = 0; j < PB_TILE; j += 8u) {
      const uint32_t p = k * PB_TILE + j;
      uint32_t cw[8], x[8], y[8], qv[8], w[4];
#pragma unroll
      for (uint32_t u = 0; u < 8u; ++u) cw[u] = nx[u];
      philox_block_keys(K, (p >> 2) + 2u, c1, read_id, 2u, nx);
      philox_block_keys(K, (p >> 2) + 3u, c1, read_id, 2u, nx + 4);
      error_words(K, read_id, c1, p, x, y);
      error_words(K, read_id, c1, p + 4u, x + 4, y + 4);
#pragma unroll
      for (uint32_t u = 0; u < 8u; ++u) {
        const uint32_t e = T.t2[row + mulhi32(cw[u] & 0xFFFF0000u, mod)];
        row = e & 0xFFFFu;
        mod = (e >> 16) & 0xFFu;
        qv[u] = T.emis[row + mulhi32(cw[u] << 16, e >> 24)];
      }
      t.prob = 0;  // 8 positions of at most 2^PB_PROB_SHIFT each
      qs_error_group(T.fast, qv, x, y, w[0], w[1], t);
      qs_error_group(T.fast, qv + 4, x + 4, y + 4, w[2], w[3], t);
      prob += t.prob;
      store_u16x8(slot + j, w);
    }
    if (t.big) {
      uint8_t q[PB_TILE];
      for (uint32_t j = 0; j < PB_TILE; ++j) q[j] = (uint8_t)(slot[j] & 0x7Fu);
      qshmm_segment_generic(T, K, read_id, pass, k * PB_TILE, k == 0, q, slot, res[k]);
      continue;
    }
    if (k == 0) t.ndel -= qs_fix_leading(T, K, read_id, c1, slot);
    SegResult r;
    r.n_entries = PB_TILE;
    r.ref_adv = PB_TILE - t.nins + t.ndel;
    r.nsub = t.nsub;
    r.ndel = t.ndel;
    r.flags = 0;
    r.pad = 0;
    r.prob = prob;
    res[k] = r;
  }
}

// Reference bases after which no deletion can follow: in the default bias mode hp_del_bias[hp] is 1 for hp 1..10
// and 0 for the cells the reference reads out of bounds (hp 11, i.e. homopolymers >= 11; DESIGN.md quirks), so the
// effect of the homopolymer table on a read is exactly "a deletion run stops in front of such a base".  Segments are
// simulated without knowing their reference offset; the walk below, which does know it, repairs those runs.
struct HpProbe {
  uint32_t enabled;         // 0: the read touches no exceptional block, nothing to repair
  WindowRef win;
  const uint32_t *xm;       // 1 bit per 1024-base block holding an exceptional base
  const uint8_t *bias_one;  // [12] hp_del_bias[h] == 1
  PB_HD bool suppress(uint32_t r_prev) const {
    const uint32_t g = win.gidx(r_prev);
    const uint32_t blk = g >> 10;
    if (((xm[blk >> 5] >> (blk & 31u)) & 1u) == 0u) return false;
    return bias_one[win.hp(r_prev)] == 0;
  }
};

struct TileWalk {
  uint32_t n_entries, positions, ref_adv, nsub, ndel;
  uint32_t ended;           // the reference window was used up inside this tile
  uint64_t prob;            // fixed-point sum of the error probabilities of the positions walked
};

// Walk the entries of one tile knowing the reference offset it starts at: stop where the window is used up
// (`while (ref_offset < mut.len)`, :2213 and :2268), clip the last deletion run, and (HpProbe) cut deletion runs
// in front of suppressing bases.  Entries are rewritten in place; entries after the end are not counted.
// p_left (--method sample): read positions left before the read is as long as its quality string; that last position
// draws no deletion and ends the read (`while (ref_offset < len && read_offset < len)`, :1775-1833).
PB_HD TileWalk qshmm_walk_tile(uint16_t *ev, uint32_t n_entries, uint32_t R_start, uint32_t wlen,
                               const QsFast *fast, const HpProbe &hp, uint32_t *blocked_io = nullptr,
                               uint32_t p_left = 0xFFFFFFFFu) {
  TileWalk t;
  t.n_entries = 0; t.positions = 0; t.ref_adv = 0; t.nsub = 0; t.ndel = 0; t.ended = 0; t.prob = 0;
  uint32_t R = R_start;
  // the current deletion run has ended (window end or suppressing base); carried between calls when a tile is
  // walked in pieces, because continuation entries of that run may follow in the next piece
  bool blocked = blocked_io ? (*blocked_io != 0u) : false;
  for (uint32_t i = 0; i < n_entries; ++i) {
    const uint32_t v = ev[i];
    const uint32_t kind = (v >> 7) & 3u;
    const bool cont = kind == 3u;
    const uint32_t part = cont ? ((v & 0x7Fu) | ((v >> 9) << 7)) : (v >> 12);
    bool last_position = false;
    if (!cont) {
      if (R >= wlen || t.positions >= p_left) { t.ended = 1; break; }
      t.prob += fast[v & 0x7Fu].prob;
      t.positions += 1u;
      t.nsub += (kind == PB_KIND_SUB) ? 1u : 0u;
      R += (kind == PB_KIND_INS) ? 0u : 1u;
      blocked = false;
      if (t.positions == p_left) blocked = last_position = true;
    }
    uint32_t take = 0;
    if (!blocked) {
      const uint32_t room = wlen - R;
      uint32_t lim = part < room ? part : room;
      if (hp.enabled) {
        for (uint32_t j = 0; j < lim; ++j) {
          if (R + j != 0u && hp.suppress(R + j - 1u)) { lim = j; break; }
        }
      }
      take = lim;
      if (take < part) blocked = true;
    }
    if (take != part) {
      if (cont) ev[i] = (uint16_t)((take & 0x7Fu) | (3u << 7) | ((take >> 7) << 9));
      else ev[i] = (uint16_t)((v & 0x0FFFu) | (take << 12));
    }
    t.ndel += take;
    R += take;
    t.n_entries = i + 1u;
    if (R >= wlen || last_position) { t.ended = 1; break; }
  }
  t.ref_adv = R - R_start;
  if (blocked_io) *blocked_io = blocked ? 1u : 0u;
  return t;
}

// Combine the segments of one read: prefix over the per-segment totals, find the segment in which the window
// is used up, clip it, write the tile checkpoints (pad = entries of the tile) and the read's totals.
// flags: 1 slot overflow, 2 coupling failed, 4 not enough segments provisioned, 8 a later segment started
// at reference offset 0 (the hp[-1] rule would apply there) -> the engine redoes the batch sequentially.
struct SegRead {
  uint32_t n_tiles, rlen, ncol, nsub, nins, ndel, flags;
  double accuracy;
};

// provisioned segments: expected positions (rho per reference base) + 1.5 % + 8 sqrt(wlen) + 64 of headroom.
// Under-provisioning is detected (flag 4) and the engine redoes the batch without segments.
PB_HD uint32_t qshmm_segments_for(uint32_t wlen, float rho) {
  const double need = (double)wlen * (double)rho * 1.015 + 8.0 * sqrt((double)wlen) + 64.0;
  return (uint32_t)((need + (double)(PB_TILE - 1u)) / (double)PB_TILE);
}

// p_len (--method sample): the read also ends when it is p_len positions long (its quality string; k_find_end's
// `sample` rule).
PB_HD void qshmm_finish_segmented(uint16_t *ev_base, const SegResult *seg, uint32_t n_seg, uint32_t wlen,
                                  const QsFast *fast, const HpProbe &hp, Ckpt *ck, SegRead &out,
                                  uint32_t p_len = 0xFFFFFFFFu) {
  uint32_t R = 0, P = 0, D = 0, nsub = 0;
  uint64_t prob = 0;
  out.flags = 0;
  out.n_tiles = 0;
  bool done = false;
  for (uint32_t k = 0; k < n_seg && !done; ++k) {
    out.flags |= seg[k].flags;
    if (k >= 1u && R == 0u) out.flags |= 8u;
    Ckpt c; c.col = P + D; c.ref = R; c.read = P; c.pad = seg[k].n_entries;
    const bool may_end = (uint64_t)R + seg[k].ref_adv >= wlen || (uint64_t)(k + 1u) * PB_TILE >= p_len;
    if (may_end || hp.enabled) {
      // exact walk: the last tile of every read, and every tile of a read that may need deletion-run repairs
      const TileWalk t = qshmm_walk_tile(ev_base + (uint64_t)k * PB_SEG_STRIDE, seg[k].n_entries, R, wlen, fast, hp, nullptr,
                                         p_len == 0xFFFFFFFFu ? 0xFFFFFFFFu : p_len - P);
      c.pad = t.n_entries;
      P += t.positions; R += t.ref_adv; D += t.ndel; nsub += t.nsub;
      prob += t.ended ? t.prob : seg[k].prob;  // a full tile's sum is the segment's own (same order, same value)
      if (t.ended) {
        out.n_tiles = k + 1u;
        done = true;
      }
    } else {
      P += PB_TILE; R += seg[k].ref_adv; D += seg[k].ndel; nsub += seg[k].nsub; prob += seg[k].prob;
    }
    ck[k] = c;
  }
  if (!done) out.flags |= 4u;
  out.rlen = P;
  out.ncol = P + D;
  out.nsub = nsub;
  out.ndel = D;
  out.nins = P + D - R;
  out.accuracy = 1.0 - (((double)prob / (double)(1u << PB_PROB_SHIFT)) / (double)P);
}

// ---------------------------------------------------------------------------------------------
// errhmm
// ---------------------------------------------------------------------------------------------
// Tables of the accuracy that drives the chain (the read's own, or the model's nearest one):
//   t2[s*1000 + k]  : next state | modulus(next state) << 6 ; row 0 is init2state
//   emis[s*1000 + k]: 0 match, 1 substitution, 2 insertion ; emod[s] its modulus (0: uniform %3)
//   edel[s]         : max over hp of floor(emis2del[s] * hp_del_bias[hp])  (1..1000 scale)
//   edel_hp[s*12+h] : exact floor(emis2del[s] * hp_del_bias[h])
//   mode            : 0 modelled accuracy, 1 below the model range (errors added, :3892-3899),
//                     2 above it (errors removed, :3920-3925), 3 accuracy 100: verbatim copy (:3837)
struct ErView {
  const uint16_t *t2;
  const uint8_t *emis;
  const uint16_t *emod;
  const uint16_t *edel;
  const uint16_t *edel_hp;
  uint32_t init_mod, mode, rate_mag;
};

struct ErSink {
  uint8_t *ev;
  Ckpt *ck;
  uint32_t n, cap;
  uint64_t acc;
  PB_HD void init(uint8_t *e, Ckpt *c, uint32_t capacity) { ev = e; ck = c; n = 0; cap = capacity; acc = 0; }
  PB_HD bool full() const { return n + 1u > cap; }
  PB_HD void checkpoint(uint32_t col, uint32_t ref, uint32_t read) {
    if ((n & (PB_TILE - 1u)) == 0u) {
      Ckpt c; c.col = col; c.ref = ref; c.read = read; c.pad = 0;
      ck[n / PB_TILE] = c;
    }
  }
  PB_HD void push(uint32_t e) {
    acc |= (uint64_t)e << (8u * (n & 7u));
    ++n;
    if ((n & 7u) == 0u) {
      *reinterpret_cast<uint64_t *>(ev + n - 8u) = acc;
      acc = 0;
    }
  }
  PB_HD void flush() {
    const uint32_t rem = n & 7u;
    for (uint32_t i = 0; i < rem; ++i) ev[n - rem + i] = (uint8_t)(acc >> (8u * i));
  }
};

// ---------------------------------------------------------------------------------------------
// errhmm SEGMENT-PARALLEL pass 1 (PHILOX).  Same idea as for qshmm; a segment is PB_TILE alignment columns and
// every column is exactly one entry, so the tiles of a read stay one contiguous stream.  Start states always come
// from the chain-only prepass.  A column whose deletion test succeeded also records what it would have been had
// the homopolymer table suppressed the deletion (bits 5-6, flag bit 7), so that the walk that knows the reference
// offset can repair it without tables:   entry = kind | info << 2 | alt_kind << 5 | deletion-test flag << 7
// ---------------------------------------------------------------------------------------------
PB_HD uint32_t er_apply_mag(uint32_t kind, uint32_t mode, uint32_t rate_mag, uint32_t mag, uint32_t mag3) {
  if (mode == 1u) return (kind == PB_KIND_MATCH && mag <= rate_mag) ? mag3 : kind;       // :3892-3899
  if (mode == 2u) return (kind != PB_KIND_MATCH && mag <= rate_mag) ? PB_KIND_MATCH : kind;  // :3920-3925
  return kind;
}

// Exact chain state in front of column c_target, computed from column 0.  While no read base has been produced
// the init row is drawn again at every column (:3853), so the leading columns are evaluated completely (deletion
// test included); after the first read base only the chain advances.  `rec`, if given, receives
// state | modulus << 6 | "no read base yet" << 31 in front of every segment k >= 1 passed on the way.
PB_HD void errhmm_state_at(const ErView &T, const PhiloxKeys &K, const HpProbe &hp, uint32_t read_id, uint32_t pass,
                           uint32_t c_target, uint32_t &state_out, uint32_t &mod_out, bool &pzero_out, uint32_t *rec) {
  uint32_t state = 0, mod = T.init_mod;
  const uint32_t c1 = pass << 16;
  uint32_t cw[4] = {0, 0, 0, 0};
  bool pzero = true;
  uint32_t c = 0;
  // phase 1: column by column until the first read base exists (init row, :3853) and the column index is a
  // multiple of 4 again
  for (; c < c_target && (pzero || (c & 3u) != 0u); ++c) {
    if (c == 0u || (c & 3u) == 0u) philox_block_keys(K, c >> 2, c1, read_id, 2u, cw);
    const uint32_t k4 = c & 3u;
    const uint32_t wdraw = k4 == 0u ? cw[0] : (k4 == 1u ? cw[1] : (k4 == 2u ? cw[2] : cw[3]));
    const uint32_t row = pzero ? 0u : state;
    const uint32_t m = pzero ? T.init_mod : mod;
    const uint32_t t = T.t2[row * PB_ER_ROW + mulhi32(wdraw, m)];
    state = t & 63u;
    mod = t >> 6;
    if (pzero) {
      // does this column produce a read base?  (reference offset == column index while only deletions came)
      uint32_t w[4];
      philox_block_keys(K, c, c1, read_id, 1u, w);
      const uint32_t x = mulhi32(w[1], 1000u) + 1u;
      bool isdel = x <= T.edel[state];
      if (isdel && hp.enabled && hp.suppress(c)) isdel = false;
      const uint32_t em = T.emod[state];
      const uint32_t k2 = (em == 0u) ? mulhi32(w[2], 3u) : (uint32_t)T.emis[state * PB_ER_ROW + mulhi32(w[2], em == 0u ? 1u : em)];
      const uint32_t mag = mulhi32(w[3], 100u) + 1u, mag3 = (((w[3] & 0xFFFu) * 3u) >> 12) + 1u;
      const uint32_t kind = er_apply_mag(isdel ? PB_KIND_DEL : k2, T.mode, T.rate_mag, mag, mag3);
      if (kind != PB_KIND_DEL) pzero = false;
    }
    if (rec && ((c + 1u) & (PB_TILE - 1u)) == 0u) rec[(c + 1u) / PB_TILE] = state | (mod << 6) | (pzero ? 0x80000000u : 0u);
  }
  // phase 2: transition rows only, four columns per step; the next block of chain draws is computed while the
  // dependent lookups of the current one run
  if (c + 4u <= c_target) {
    uint32_t nx[4];
    philox_block_keys(K, c >> 2, c1, read_id, 2u, nx);
    for (; c + 4u <= c_target; c += 4u) {
      const uint32_t w4[4] = {nx[0], nx[1], nx[2], nx[3]};
      philox_block_keys(K, (c >> 2) + 1u, c1, read_id, 2u, nx);
#pragma unroll
      for (uint32_t u = 0; u < 4u; ++u) {
        const uint32_t t = T.t2[state * PB_ER_ROW + mulhi32(w4[u], mod)];
        state = t & 63u;
        mod = t >> 6;
      }
      if (rec && ((c + 4u) & (PB_TILE - 1u)) == 0u) rec[(c + 4u) / PB_TILE] = state | (mod << 6);
    }
  }
  // tail: fewer than four columns left
  if (c < c_target) {
    philox_block_keys(K, c >> 2, c1, read_id, 2u, cw);
    for (; c < c_target; ++c) {
      const uint32_t k4 = c & 3u;
      const uint32_t wdraw = k4 == 0u ? cw[0] : (k4 == 1u ? cw[1] : (k4 == 2u ? cw[2] : cw[3]));
      const uint32_t t = T.t2[state * PB_ER_ROW + mulhi32(wdraw, mod)];
      state = t & 63u;
      mod = t >> 6;
    }
  }
  state_out = state;
  mod_out = mod;
  pzero_out = pzero;
}

// transition rows only (a read base exists): columns [c_from, c_to), both multiples of PB_TILE; records the state in
// front of every segment boundary passed
PB_HD void errhmm_chain_range(const ErView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass, uint32_t state,
                              uint32_t mod, uint32_t c_from, uint32_t c_to, uint32_t *rec) {
  const uint32_t c1 = pass << 16;
  uint32_t nx[4];
  philox_block_keys(K, c_from >> 2, c1, read_id, 2u, nx);
  for (uint32_t c = c_from; c + 4u <= c_to; c += 4u) {
    const uint32_t w4[4] = {nx[0], nx[1], nx[2], nx[3]};
    philox_block_keys(K, (c >> 2) + 1u, c1, read_id, 2u, nx);
#pragma unroll
    for (uint32_t u = 0; u < 4u; ++u) {
      const uint32_t t = T.t2[state * PB_ER_ROW + mulhi32(w4[u], mod)];
      state = t & 63u;
      mod = t >> 6;
    }
    if (((c + 4u) & (PB_TILE - 1u)) == 0u) rec[(c + 4u) / PB_TILE] = state | (mod << 6);
  }
}

// Chain-only prepass (sticky chains): states in front of every segment k >= 1
PB_HD void errhmm_chain_only(const ErView &T, const PhiloxKeys &K, const HpProbe &hp, uint32_t read_id,
                             uint32_t pass, uint32_t n_seg, uint32_t *seg_state) {
  uint32_t st, md;
  bool pz;
  errhmm_state_at(T, K, hp, read_id, pass, (n_seg - 1u) * PB_TILE, st, md, pz, seg_state);
}

// Backward coupling for errhmm: state entering column c_start (>= PB_TILE), assuming a read base exists before the
// window (transition rows only).  A window never reaches below column 512 (then the exact walk from column 0 is
// taken instead); segment 0 reports reads whose first read base comes later than that (flag 32 -> sequential
// redo), so the assumption is checked, not hoped for.
PB_HD void errhmm_segment_start(const ErView &T, const uint16_t *tmodv, uint64_t reach, const PhiloxKeys &K,
                                const HpProbe &hp, uint32_t read_id, uint32_t pass, uint32_t c_start,
                                uint32_t first_window, uint32_t &state, uint32_t &mod, bool &pzero) {
  const uint32_t c1 = pass << 16;
  for (uint32_t B = first_window;; B *= 2u) {
    if (c_start < B + 512u) {
      errhmm_state_at(T, K, hp, read_id, pass, c_start, state, mod, pzero, nullptr);
      return;
    }
    const uint32_t c0 = c_start - B;
    uint64_t mask = reach;
    uint32_t s_state = 0, s_mod = 1;
    bool single = false;
    uint32_t cwb[4] = {0, 0, 0, 0};
    for (uint32_t c = c0; c < c_start; ++c) {
      if (c == c0 || (c & 3u) == 0u) philox_block_keys(K, c >> 2, c1, read_id, 2u, cwb);
      const uint32_t k4 = c & 3u;
      const uint32_t wdraw = k4 == 0u ? cwb[0] : (k4 == 1u ? cwb[1] : (k4 == 2u ? cwb[2] : cwb[3]));
      if (single) {
        const uint32_t t = T.t2[s_state * PB_ER_ROW + mulhi32(wdraw, s_mod)];
        s_state = t & 63u;
        s_mod = t >> 6;
      } else {
        uint64_t next = 0;
        uint32_t last_t = 0;
        for (uint64_t m = mask; m; m &= m - 1ull) {
#if defined(__CUDA_ARCH__)
          const uint32_t s = (uint32_t)__ffsll((long long)m) - 1u;
#else
          const uint32_t s = (uint32_t)__builtin_ctzll(m);
#endif
          last_t = T.t2[s * PB_ER_ROW + mulhi32(wdraw, tmodv[s])];
          next |= 1ull << (last_t & 63u);
        }
        mask = next;
        if ((mask & (mask - 1ull)) == 0ull) {
          single = true;
          s_state = last_t & 63u;
          s_mod = last_t >> 6;
        }
      }
    }
    if (single) {
      state = s_state;
      mod = s_mod;
      pzero = false;
      return;
    }
  }
}

PB_HD void errhmm_simulate_segment(const ErView &T, const PhiloxKeys &K, uint32_t read_id, uint32_t pass,
                                   uint32_t c_start, bool pzero_in, uint32_t state, uint32_t mod, uint8_t *ev,
                                   SegResult &res) {
  uint32_t radv = 0, nsub = 0, ndel = 0, nins = 0;
  bool late = false;
  bool pzero = pzero_in;  // no read base yet: the init row is drawn again (:3853)
  const uint32_t c1 = pass << 16;
  for (uint32_t C = c_start; C < c_start + PB_TILE; C += PB_GROUP) {
    uint32_t g[PB_GROUP][4], cw[PB_GROUP];
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) philox_block_keys(K, C + u, c1, read_id, 1u, g[u]);
    philox_block_keys(K, C >> 2, c1, read_id, 2u, cw);
    uint32_t packed = 0;
#pragma unroll
    for (uint32_t u = 0; u < PB_GROUP; ++u) {
      const uint32_t w0 = g[u][0], w1 = g[u][1], w2 = g[u][2], w3 = g[u][3];
      const uint32_t row = pzero ? 0u : state;
      const uint32_t m = pzero ? T.init_mod : mod;
      const uint32_t t = T.t2[row * PB_ER_ROW + mulhi32(cw[u], m)];
      state = t & 63u;
      mod = t >> 6;
      const uint32_t x = mulhi32(w1, 1000u) + 1u;
      const bool isdel = x <= T.edel[state];
      const uint32_t em = T.emod[state];
      const uint32_t k2 = (em == 0u) ? mulhi32(w2, 3u) : (uint32_t)T.emis[state * PB_ER_ROW + mulhi32(w2, em == 0u ? 1u : em)];
      const uint32_t mag = mulhi32(w3, 100u) + 1u, mag3 = (((w3 & 0xFFFu) * 3u) >> 12) + 1u;
      const uint32_t kind = er_apply_mag(isdel ? PB_KIND_DEL : k2, T.mode, T.rate_mag, mag, mag3);
      const uint32_t alt = er_apply_mag(k2, T.mode, T.rate_mag, mag, mag3);
      const uint32_t c3 = ((w0 & 0xFFFu) * 3u) >> 12, c8 = w1 & 7u;
      const uint32_t info = kind == PB_KIND_SUB ? c3 : (kind == PB_KIND_INS ? c8 : 0u);
      const uint32_t e = kind | (info << 2) | (isdel ? ((alt << 5) | 0x80u) : 0u);
      packed |= e << (8u * u);
      nsub += (kind == PB_KIND_SUB) ? 1u : 0u;
      nins += (kind == PB_KIND_INS) ? 1u : 0u;
      ndel += (kind == PB_KIND_DEL) ? 1u : 0u;
      radv += (kind == PB_KIND_INS) ? 0u : 1u;
      if (kind != PB_KIND_DEL) pzero = false;
    }
    *reinterpret_cast<uint32_t *>(ev + (C - c_start)) = packed;
    if (pzero && C - c_start + PB_GROUP >= 512u) late = true;
  }
  res.n_entries = PB_TILE;
  res.ref_adv = radv;
  res.nsub = nsub;
  res.ndel = ndel;
  res.flags = (late && pzero_in) ? 32u : 0u;  // no read base in the first 512 columns: coupling assumptions void
  res.pad = 0;
  res.prob = nins;               // errhmm: the insertion count travels in the otherwise unused field
}

struct ErTileWalk {
  uint32_t n_entries, positions, ref_adv, nsub, nins, ndel, ended;
  uint32_t early_repair;  // a suppressed deletion before the first read base: init-row bookkeeping is off -> redo
};

// exact walk of columns [0, n) of a tile that starts at reference offset R_start: stops where the window is used up
// (:3850) and, for reads touching exceptional blocks, turns deletion columns that the homopolymer table suppresses
// (hp at the CURRENT base, :3860) into their recorded alternative
PB_HD ErTileWalk errhmm_walk_tile(uint8_t *ev, uint32_t n, uint32_t R_start, uint32_t P_start, uint32_t wlen,
                                  const HpProbe &hp, const PhiloxKeys &K, uint32_t read_id, uint32_t pass,
                                  uint32_t c_abs) {
  ErTileWalk t;
  t.n_entries = 0; t.positions = 0; t.ref_adv = 0; t.nsub = 0; t.nins = 0; t.ndel = 0; t.ended = 0; t.early_repair = 0;
  uint32_t R = R_start;
  for (uint32_t i = 0; i < n; ++i) {
    if (R >= wlen) { t.ended = 1; break; }
    uint32_t v = ev[i];
    uint32_t kind = v & 3u;
    if (hp.enabled && (v & 0x80u) && hp.suppress(R)) {
      if (P_start + t.positions == 0u) t.early_repair = 1u;
      kind = (v >> 5) & 3u;
      uint32_t w[4];
      philox_block_keys(K, c_abs + i, pass << 16, read_id, 1u, w);
      const uint32_t info = kind == PB_KIND_SUB ? (((w[0] & 0xFFFu) * 3u) >> 12) : (kind == PB_KIND_INS ? (w[1] & 7u) : 0u);
      v = kind | (info << 2);
      ev[i] = (uint8_t)v;
    }
    t.positions += (kind == PB_KIND_DEL) ? 0u : 1u;
    t.nsub += (kind == PB_KIND_SUB) ? 1u : 0u;
    t.nins += (kind == PB_KIND_INS) ? 1u : 0u;
    t.ndel += (kind == PB_KIND_DEL) ? 1u : 0u;
    R += (kind == PB_KIND_INS) ? 0u : 1u;
    t.n_entries = i + 1u;
    if (R >= wlen) { t.ended = 1; break; }
  }
  t.ref_adv = R - R_start;
  return t;
}

// sequential statement of the errhmm find_end (the GPU runs a warp-cooperative version, seg_kernels.cuh)
PB_HD void errhmm_finish_segmented(uint8_t *ev_base, const SegResult *seg, uint32_t n_seg, uint32_t wlen,
                                   const HpProbe &hp, const PhiloxKeys &K, uint32_t read_id, uint32_t pass, Ckpt *ck,
                                   SegRead &out) {
  uint32_t R = 0, P = 0, nsub = 0, nins = 0, ndel = 0, C = 0;
  out.flags = 0;
  out.n_tiles = 0;
  bool done = false;
  for (uint32_t k = 0; k < n_seg && !done; ++k) {
    out.flags |= seg[k].flags;
    Ckpt c; c.col = C; c.ref = R; c.read = P; c.pad = PB_TILE;
    ck[k] = c;
    if (hp.enabled || (uint64_t)R + seg[k].ref_adv >= wlen) {
      const ErTileWalk t = errhmm_walk_tile(ev_base + (uint64_t)k * PB_TILE, PB_TILE, R, P, wlen, hp, K, read_id, pass, k * PB_TILE);
      if (t.early_repair) out.flags |= 8u;
      P += t.positions; R += t.ref_adv; nsub += t.nsub; nins += t.nins; ndel += t.ndel; C += t.n_entries;
      if (t.ended) {
        out.n_tiles = k + 1u;
        done = true;
      }
    } else {
      const uint32_t si = (uint32_t)seg[k].prob;
      P += PB_TILE - seg[k].ndel; R += seg[k].ref_adv; nsub += seg[k].nsub; nins += si; ndel += seg[k].ndel; C += PB_TILE;
    }
  }
  if (!done) out.flags |= 4u;
  out.rlen = P;
  out.ncol = C;
  out.nsub = nsub;
  out.nins = nins;
  out.ndel = ndel;
  out.accuracy = 1.0 - ((double)(nsub + nins + ndel) / (double)P);
}

template <class Draw>
PB_HD void errhmm_simulate(const ErView &T, Draw &d, const WindowRef &win, bool slow, uint32_t wlen,
                           ErSink &sink, SubreadResult &res) {
  uint32_t R = 0, P = 0, C = 0;
  uint32_t state = 0, mod = T.init_mod;
  uint32_t nsub = 0, nins = 0, ndel = 0;
  res.overflow = 0;
  if (T.mode == 3u) {
    while (R < wlen) {
      if (sink.full()) { res.overflow = 1; break; }
      sink.checkpoint(C, R, P);
      sink.push(PB_KIND_MATCH);
      ++R; ++P; ++C;
    }
  } else {
    while (R < wlen) {
      d.prefetch(C);
#pragma unroll
      for (uint32_t u = 0; u < PB_GROUP; ++u) {
        if (R >= wlen) break;
        if (sink.full()) { res.overflow = 1; break; }
        sink.checkpoint(C, R, P);
        d.begin(u);
        const uint32_t row = (P == 0u) ? 0u : state;           // init is re-drawn while read_offset == 0 (:3853)
        const uint32_t m = (P == 0u) ? T.init_mod : mod;
        const uint32_t t = T.t2[row * PB_ER_ROW + d.wc(C, m)];
        state = t & 63u;
        mod = t >> 6;
        const uint32_t x = d.w1(1000u) + 1u;
        bool isdel = x <= T.edel[state];
        if (isdel && slow) isdel = x <= T.edel_hp[state * 12u + win.hp(R)];   // hp at the current base (:3860)
        uint32_t kind;
        if (Draw::kCounter) {
          const uint32_t em = T.emod[state];
          const uint32_t k2 = (em == 0u) ? d.w2(3u) : (uint32_t)T.emis[state * PB_ER_ROW + d.w2(em == 0u ? 1u : em)];
          kind = isdel ? PB_KIND_DEL : k2;
        } else if (isdel) {
          kind = PB_KIND_DEL;
        } else {
          const uint32_t em = T.emod[state];
          kind = (em == 0u) ? d.w2(3u) : (uint32_t)T.emis[state * PB_ER_ROW + d.w2(em)];
        }
        if (T.mode == 1u) {
          if (kind == PB_KIND_MATCH) {
            if (d.w3(100u) + 1u <= T.rate_mag) kind = d.mag3();
          }
        } else if (T.mode == 2u) {
          if (kind != PB_KIND_MATCH) {
            if (d.w3(100u) + 1u <= T.rate_mag) kind = PB_KIND_MATCH;
          }
        }
        uint32_t info = 0;
        if (Draw::kCounter) {
          info = (kind == PB_KIND_SUB) ? d.choice3() : ((kind == PB_KIND_INS) ? d.choice8() : 0u);
        } else {
          if (kind == PB_KIND_SUB) info = d.choice3();
          else if (kind == PB_KIND_INS) info = d.choice8();
        }
        if (slow && kind == PB_KIND_SUB && win.nonacgt(R)) info = d.choice4();
        nsub += (kind == PB_KIND_SUB) ? 1u : 0u;
        nins += (kind == PB_KIND_INS) ? 1u : 0u;
        ndel += (kind == PB_KIND_DEL) ? 1u : 0u;
        R += (kind == PB_KIND_INS) ? 0u : 1u;
        P += (kind == PB_KIND_DEL) ? 0u : 1u;
        ++C;
        sink.push(kind | (info << 2));
      }
      if (res.overflow) break;
    }
  }
  sink.flush();
  res.n_entries = sink.n;
  res.rlen = P;
  res.ncol = C;
  res.nsub = nsub;
  res.nins = nins;
  res.ndel = ndel;
  res.accuracy = 1.0 - ((double)(nsub + nins + ndel) / (double)P);  // :4002
}

}  // namespace pb
