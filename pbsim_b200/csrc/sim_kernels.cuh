// K1 (read planner) and K2/K3 (pass 1: qshmm / errhmm chains -> event streams).
//
// Scheduling: every (read, pass) — a "subread" — is one GPU thread in pass 1, because the Markov
// chain of a read is inherently sequential.  Subreads are sorted by (accuracy, length descending)
// so that (a) a CTA works on ONE accuracy and stages only that accuracy's HMM tables in shared
// memory with a TMA bulk copy, and (b) the 32 lanes of a warp run reads of near-equal length
// (length-binned scheduling; longest first so the tail of the grid is made of short reads).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "k0_genome.cuh"
#include "model_image.hpp"
#include "sim_core.cuh"

namespace pb {

constexpr int kSimThreads = 128;  // qshmm: sub-reads / segments per pass-1 CTA (tables: 28 KB of shared memory)
constexpr int kErrThreads = 512;  // errhmm: its 1000-resolution tables take 60-90 KB, so more threads share them
constexpr int kBins = 202;        // schedule bins: accuracy * 2 + slow  (slow reads get CTAs of their own)

struct DeviceModel {
  const uint8_t *blob;
  const AccEntry *acc;        // [101]
  const int32_t *prob2len;
  const uint8_t *prob2acc;
  uint32_t len_rand_value, acc_rand_value, len_min;
  const uint8_t *qs_tabs;     // [kQsTabBytes] thr 94*16 | qc_prob 94*8 | thr32 94*16 | fast 94*16 (one bulk copy)
  const uint32_t *qs_thr_hp;  // [94*12]
  const uint32_t *qs_thr_hp32;// [94*12] the same on the T32 scale (PHILOX mode)
  const uint32_t *qs_thr32;   // [94*4]  = qs_tabs + kQsTabThr32
  const QsFast *qs_fast;      // [94]    = qs_tabs + kQsTabFast
  const uint16_t *er_bias;
  uint32_t pass_num;
  uint32_t uniform_bias;
  uint32_t method;            // PBSIM_METHOD_*
};

struct DeviceGenome {
  const uint8_t *ascii;
  const uint32_t *pk;
  const uint8_t *hp4;
  const uint32_t *xm;
  uint32_t len;
  uint32_t seq_num;
};

// --strategy trans / templ: the sequences are concatenated into the device genome; reads are numbered through the
// whole set (sim.res_num) and belong to sequence t when rprefix[t] < read id <= rprefix[t+1]
struct DeviceSet {
  uint32_t strategy;        // PBSIM_STRATEGY_*; WGS: every pointer below is null
  uint32_t n;
  const uint32_t *start;    // [n+1] first base of sequence t in the concatenation
  const uint64_t *rprefix;  // [n+1] reads of the sequences before t (trans: plus + minus each; templ: 1 each)
  const uint32_t *plus;     // [n]   trans: the first plus[t] reads of a transcript are '+', the rest '-'
  const uint16_t *ssp_ends; // start-position table, see plan_read_trans
  const uint16_t *ssp_mod;
  const uint8_t *ids;       // names, concatenated
  const uint32_t *id_start; // [n+1]
  // replay of simulate_by_errhmm_trans only: sequence and rank of every logged read (null otherwise).  The
  // reference's read counter of a transcript jumps after an accuracy-100 read (pbsim.cpp:4487, :4532), so which reads
  // exist depends on the draws; the host works the sequence out from the log (engine.cu build_replay_read_map).
  const uint32_t *map_tr, *map_k;
};

struct RngParams {
  uint32_t mode;           // PBSIM_RNG_*
  uint32_t seed;
  const int32_t *draws;    // replay: device copy of the slice of the log this batch needs
  int64_t draws_base;      // index in the full log of draws[0]
  int64_t draws_end;       // one past the last available draw (full-log index)
  const int64_t *starts;   // replay: first draw of every subread of this batch (full-log index)
};

// per-batch arrays (device)
struct Batch {
  uint32_t n_reads, n_sub;
  uint64_t first_read;     // id of read 0 of the batch minus 1 (ids are first_read + 1 + r)
  // per read
  uint32_t *plan_off, *plan_wlen, *plan_raw, *plan_meta;  // meta: acc | minus<<8 | slow<<9 | invalid<<10
  uint32_t *plan_tr;       // sequence index of the read (trans / templ; unused for WGS)
  // per subread
  uint32_t *key_in, *key_out, *idx_in, *order;
  uint32_t *cap;           // event-slot capacity (entries)
  uint64_t *ev_off;        // exclusive scan of cap
  uint32_t *ck_cap;        // checkpoint slots
  uint64_t *ck_off;
  uint32_t *nent, *rlen, *ncol, *nsub, *nins, *ndel, *flags, *draws_used;
  uint32_t *nseg;          // segments provisioned (0: the sub-read runs on the sequential pass-1 path)
  uint32_t *nchunk;        // chain chunks: threads of k_qs_pass1 / k_chain_chunk_err that walk its segments
  double *accuracy;
  // --method sample, per read: which copy of its group (pool entry, pool pass) a read is, and the group's size
  uint32_t *grp_copy, *grp_num;
};

// ----------------------------------------------------------------------------------------------
// K1: plan.  One thread per read.  clip_room >= 0 only for single-read tail batches.
// ----------------------------------------------------------------------------------------------
template <class Draw>
__device__ __forceinline__ ReadPlan plan_any(const PlanTables &T, Draw &d, const DeviceGenome &G, const DeviceSet &S,
                                             uint32_t tlen, int64_t clip_room) {
  if (S.strategy == PBSIM_STRATEGY_TRANS) return plan_read_trans(T, d, S.ssp_ends, S.ssp_mod, tlen);
  if (S.strategy == PBSIM_STRATEGY_TEMPL) return plan_read_templ(T, d, tlen);
  return plan_read(T, d, G.len, clip_room);
}

__global__ void k_plan(DeviceModel M, DeviceGenome G, DeviceSet S, RngParams rng, Batch B, int64_t clip_room,
                       uint32_t cap_num, uint32_t cap_den, uint32_t ev_align, uint32_t seg_min_len /* 0: segments off */,
                       float seg_extra /* extra segment headroom learnt from earlier batches */,
                       uint32_t chain_chunk /* segments per chain chunk */) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= B.n_reads) return;
  PlanTables T;
  T.prob2len = M.prob2len;
  T.prob2acc = M.prob2acc;
  T.len_rand_value = M.len_rand_value;
  T.acc_rand_value = M.acc_rand_value;
  T.len_min = M.len_min;
  const uint64_t read_id = B.first_read + 1u + r;
  ReadPlan p;
  // sequence sets: which sequence the read belongs to, and its rank among that sequence's reads
  uint32_t tr = 0, tlen = 0, tstart = 0;
  uint64_t kth = 0;
  if (S.strategy != PBSIM_STRATEGY_WGS) {
    if (S.map_tr != nullptr) {
      tr = S.map_tr[read_id - 1u];
      kth = S.map_k[read_id - 1u];
    } else {
      uint32_t lo = 0, hi = S.n;  // rprefix[lo] <= read_id - 1 < rprefix[hi]
      while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (S.rprefix[mid] <= read_id - 1u) lo = mid;
        else hi = mid;
      }
      tr = lo;
      kth = read_id - S.rprefix[tr];
    }
    tstart = S.start[tr];
    tlen = S.start[tr + 1] - tstart;
    B.plan_tr[r] = tr;
  }
  if (rng.mode == PBSIM_RNG_PHILOX) {
    PhiloxDraw d;
    d.ph.k0 = rng.seed;
    d.ph.k1 = G.seq_num;
    d.read_id = (uint32_t)read_id;
    d.pass = 0;
    p = plan_any(T, d, G, S, tlen, clip_room);
  } else {
    ReplayDraw d;
    d.log = rng.draws - rng.draws_base;
    d.cur = rng.starts[(uint64_t)r * M.pass_num];
    d.start = d.cur;
    d.end = rng.draws_end;
    p = plan_any(T, d, G, S, tlen, clip_room);
  }
  p.offset += tstart;  // position in the concatenation
  uint32_t minus = (read_id & 1u) ? 0u : 1u;  // res_num odd -> '+', even -> '-' (:2201-2207)
  if (S.strategy == PBSIM_STRATEGY_TRANS) minus = kth <= S.plus[tr] ? 0u : 1u;  // i <= plus_exp -> '+' (:2880)
  if (S.strategy == PBSIM_STRATEGY_TEMPL) minus = 0u;                           // :3363
  bool slow = !M.uniform_bias;
  if (!slow) slow = range_exceptional(G.xm, p.offset, p.offset + p.wlen - 1u);
  const AccEntry ae = M.acc[p.acc];
  B.plan_off[r] = p.offset;
  B.plan_wlen[r] = p.wlen;
  B.plan_raw[r] = p.raw_len;
  // segment-parallel pass 1: PHILOX-mode reads of at least seg_min_len positions
  // (reads touching exceptional blocks qualify too in the default bias mode: k_find_end repairs their deletion
  // runs with the exact reference offset, pass 2 re-derives choices on non-ACGT bases)
  const bool errm = M.method == PBSIM_METHOD_ERRHMM;
  const bool segmented = seg_min_len != 0u && rng.mode == PBSIM_RNG_PHILOX && (!slow || M.uniform_bias) && ae.valid &&
                         p.wlen >= seg_min_len && !(errm && ae.mode == 3u);
  // The HMM state in front of every segment comes from chain chunks (k_qs_pass1, k_chain_chunk_err): a thread per
  // CHUNK of chain_chunk segments starts from the exact state recovered by backward coupling at the chunk's first
  // position (position 0: the init draw) and walks the chain through the chunk.  Chains with sticky states do not
  // couple quickly: their reads are one chunk.
  const bool needs_chain = segmented && (errm || ae.has_model);
  const uint32_t nseg = segmented ? qshmm_segments_for(p.wlen, ae.rho * (1.0f + seg_extra)) : 0u;
  B.plan_meta[r] = p.acc | (minus << 8) | ((slow ? 1u : 0u) << 9) | ((ae.valid ? 0u : 1u) << 10) |
                   ((segmented ? 1u : 0u) << 11) | ((needs_chain ? 1u : 0u) << 12);
  // event-slot capacity: wlen * cap_num/cap_den + slack, rounded so that slots stay 16-byte aligned
  uint64_t cap = (uint64_t)p.wlen * cap_num / cap_den + 2048u;
  if (segmented) cap = (uint64_t)nseg * (errm ? PB_TILE : PB_SEG_STRIDE) + 64u;
  cap = (cap + ev_align - 1u) / ev_align * ev_align;
  const uint32_t ckc = segmented ? nseg + 2u : (uint32_t)(cap / PB_TILE) + 2u;
  // qshmm's k_qs_pass1 walks EVERY provisioned segment (it writes the events of every position)
  uint32_t nchunk = 0;
  if (needs_chain && nseg > 0u) nchunk = ae.seg_ok ? (nseg + chain_chunk - 1u) / chain_chunk : 1u;
  for (uint32_t h = 0; h < M.pass_num; ++h) {
    const uint32_t s = r * M.pass_num + h;
    B.nchunk[s] = nchunk;
    // segmented sub-reads get the out-of-range bin kBins: the sequential schedule skips them
    B.key_in[s] = segmented ? ((uint32_t)kBins << 20)
                            : ((p.acc << 21) | ((slow ? 1u : 0u) << 20) | (0xFFFFFu - (p.wlen > 0xFFFFFu ? 0xFFFFFu : p.wlen)));
    B.idx_in[s] = s;
    B.cap[s] = (uint32_t)cap;
    B.ck_cap[s] = ckc;
    B.nseg[s] = nseg;
  }
}

// accuracy-bin boundaries in the sorted order, then the CTA map
__global__ void k_bin_bounds(const uint32_t *key_sorted, uint32_t n, uint32_t *bin_start /*[kBins]*/) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t a = key_sorted[i] >> 20;
  if (i == 0 || (key_sorted[i - 1] >> 20) != a) bin_start[a] = i;
}

// cta_first[b] = first pass-1 CTA of bin b; cta_first[kBins] = total
__global__ void k_cta_map(const uint32_t *bin_start, const uint32_t *key_sorted, uint32_t n, uint32_t *bin_lo,
                          uint32_t *bin_hi, uint32_t *cta_first, uint32_t cta_threads) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  // bin_start holds 0xFFFFFFFF for empty bins; bin kBins collects the sub-reads that are NOT scheduled here
  // (segment-parallel pass 1), they sort behind every real bin
  uint32_t next_lo = (bin_start[kBins] != 0xFFFFFFFFu) ? bin_start[kBins] : n, total = 0;
  for (int a = kBins - 1; a >= 0; --a) {
    const uint32_t lo = bin_start[a];
    if (lo == 0xFFFFFFFFu) {
      bin_lo[a] = bin_hi[a] = 0;
    } else {
      bin_lo[a] = lo;
      bin_hi[a] = next_lo;
      next_lo = lo;
    }
  }
  for (int a = 0; a < kBins; ++a) {
    cta_first[a] = total;
    total += (bin_hi[a] - bin_lo[a] + cta_threads - 1) / cta_threads;
  }
  cta_first[kBins] = total;
}

// Global longest-first dispatch: CTA b of the (bin-ordered) map gets the key "longest read it holds"
// (low 20 bits of the sort key, smaller = longer); the engine sorts CTAs by it and pass 1 runs
// CTA cta_order[blockIdx.x].  Slots beyond the map get the largest key and exit immediately.
__global__ void k_cta_keys(const uint32_t *key_sorted, const uint32_t *bin_lo, const uint32_t *cta_first,
                           uint32_t n_slots, uint32_t *cta_key, uint32_t *cta_id, uint32_t cta_threads) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_slots) return;
  cta_id[b] = b;
  if (b >= cta_first[kBins]) {
    cta_key[b] = 0x100000u;
    return;
  }
  uint32_t lo = 0, hi = kBins;  // largest bin a with cta_first[a] <= b
  while (hi - lo > 1u) {
    const uint32_t mid = (lo + hi) >> 1;
    if (cta_first[mid] <= b) lo = mid; else hi = mid;
  }
  // empty bins share cta_first with their successor: step to the last bin that starts at or before b
  const uint32_t first = bin_lo[lo] + (b - cta_first[lo]) * cta_threads;
  cta_key[b] = key_sorted[first] & 0xFFFFFu;
}

// ----------------------------------------------------------------------------------------------
// TMA (bulk async copy) staging of tables into shared memory
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// which accuracy bin does this CTA serve?  returns false if the CTA is beyond the map
__device__ __forceinline__ bool cta_assignment(const uint32_t *cta_order, const uint32_t *cta_first,
                                               const uint32_t *bin_lo, const uint32_t *bin_hi,
                                               uint32_t *acc, uint32_t *lo, uint32_t *hi) {
  __shared__ uint32_t s_acc, s_lo, s_hi, s_ok;
  if (threadIdx.x == 0) {
    const uint32_t b = cta_order[blockIdx.x];
    s_ok = 0;
    if (b < cta_first[kBins]) {
      // the last bin whose first CTA is <= b (cta_first is non-decreasing; empty bins repeat a value): binary search,
      // 8 dependent loads instead of a walk over up to kBins of them in front of every CTA's barrier
      uint32_t a = 0, top = kBins;
      while (top - a > 1u) {
        const uint32_t mid = (a + top) >> 1;
        if (cta_first[mid] <= b) a = mid;
        else top = mid;
      }
      const uint32_t local = b - cta_first[a];
      s_acc = a >> 1;
      s_lo = bin_lo[a] + local * blockDim.x;
      s_hi = min(bin_hi[a], s_lo + blockDim.x);
      s_ok = 1;
    }
  }
  __syncthreads();
  *acc = s_acc;
  *lo = s_lo;
  *hi = s_hi;
  return s_ok != 0;
}

struct SimArgs {
  PhiloxKeys keys;  // round keys of (seed, sequence): constant-bank operands of the fast path
  DeviceModel M;
  DeviceGenome G;
  RngParams rng;
  Batch B;
  const uint32_t *cta_order, *cta_first, *bin_lo, *bin_hi;
  const uint8_t *bias_one;  // [12] hp_del_bias[h] == 1
  uint32_t plan_draws;      // replay: planner draws in front of pass 0 (0: WGS, 2 or 3; trans 3; templ 1)
  uint8_t *ev;   // event arena
  Ckpt *ck;      // checkpoint arena
};

__device__ __forceinline__ void store_result(const Batch &B, uint32_t s, const SubreadResult &res, uint32_t used) {
  B.nent[s] = res.n_entries;
  B.rlen[s] = res.rlen;
  B.ncol[s] = res.ncol;
  B.nsub[s] = res.nsub;
  B.nins[s] = res.nins;
  B.ndel[s] = res.ndel;
  B.flags[s] = res.overflow;
  B.draws_used[s] = used;
  B.accuracy[s] = res.accuracy;
}

// chain draws of subread (r, h) in replay mode start after the planner's draws for pass 0: WGS 2 or 3 (:2174-2189),
// transcripts 3 (:2842-2850), templates 1 (:3359)
__device__ __forceinline__ void replay_setup(ReplayDraw &d, const RngParams &rng, uint32_t s, uint32_t pass,
                                             uint32_t fixed, bool offset_drawn) {
  d.log = rng.draws - rng.draws_base;
  d.start = rng.starts[s];
  d.cur = d.start + (pass == 0 ? (fixed ? fixed : (offset_drawn ? 3u : 2u)) : 0u);
  d.end = rng.draws_end;
}

// ----------------------------------------------------------------------------------------------
// K2: qshmm pass 1
// shared memory: [table blob | thr 94*16 | qc_prob 94*8 | mbarrier]
// ----------------------------------------------------------------------------------------------
// the per-quality tables travel as one block (DeviceModel::qs_tabs): thr | qc_prob | thr32 | fast
constexpr uint32_t kQsTabThr = 0;
constexpr uint32_t kQsTabProb = kQsTabThr + PBSIM_NQV * 16;
constexpr uint32_t kQsTabThr32 = kQsTabProb + PBSIM_NQV * 8;
constexpr uint32_t kQsTabFast = kQsTabThr32 + PBSIM_NQV * 16;
constexpr uint32_t kQsTabBytes = kQsTabFast + PBSIM_NQV * 16;
static_assert(kQsTabBytes % 16 == 0, "bulk copy size");
constexpr uint32_t kQsSmemThr = QsBlobLayout::bytes;
constexpr uint32_t kQsSmemProb = kQsSmemThr + kQsTabProb;
constexpr uint32_t kQsSmemThr32 = kQsSmemThr + kQsTabThr32;
constexpr uint32_t kQsSmemFast = kQsSmemThr + kQsTabFast;
constexpr uint32_t kQsSmemBar = kQsSmemThr + kQsTabBytes;
constexpr uint32_t kQsSmemBytes = kQsSmemBar + 16;

template <int RNG_MODE>
__global__ void __launch_bounds__(kSimThreads) k_sim_qshmm(SimArgs A) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  const AccEntry ae = A.M.acc[acc];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kQsSmemBar);
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, ae.blob_bytes + kQsTabBytes);
    tma_bulk_g2s(smem, A.M.blob + ae.blob_off, ae.blob_bytes, bar);
    tma_bulk_g2s(smem + kQsSmemThr, A.M.qs_tabs, kQsTabBytes, bar);
  }
  mbar_wait(bar, 0);

  const uint32_t k = lo + threadIdx.x;
  if (k >= hi) return;
  const uint32_t s = A.B.order[k];
  const uint32_t r = s / A.M.pass_num, pass = s % A.M.pass_num;
  const uint32_t meta = A.B.plan_meta[r];
  const uint32_t wlen = A.B.plan_wlen[r];
  if (meta & (1u << 10)) {  // accuracy without tables: flagged, reported by the host
    SubreadResult z = {};
    z.overflow = 2;
    store_result(A.B, s, z, 0);
    return;
  }
  QsView T;
  T.t2 = reinterpret_cast<const uint32_t *>(smem + QsBlobLayout::t2_off);
  T.emis = smem + QsBlobLayout::emis_off;
  T.freq = smem;
  T.has_model = ae.has_model;
  T.init_mod = ae.init_mod;
  T.freq_mod = ae.freq_mod;
  T.thr = reinterpret_cast<const QsThr *>(smem + kQsSmemThr);
  T.thr_hp = A.M.qs_thr_hp;
  T.qc_prob = reinterpret_cast<const double *>(smem + kQsSmemProb);
  T.thr32 = reinterpret_cast<const QsThr *>(smem + kQsSmemThr32);
  T.thr_hp32 = A.M.qs_thr_hp32;
  T.fast = reinterpret_cast<const QsFast *>(smem + kQsSmemFast);
  WindowRef win;
  win.ascii = A.G.ascii;
  win.hp4 = A.G.hp4;
  win.offset = A.B.plan_off[r];
  win.wlen = wlen;
  win.minus = (meta >> 8) & 1u;
  const bool slow = (meta >> 9) & 1u;
  QsSink sink;
  sink.init(reinterpret_cast<uint16_t *>(A.ev) + A.B.ev_off[s], A.ck + A.B.ck_off[s], A.B.cap[s]);
  SubreadResult res;
  uint32_t used = 0;
  if (RNG_MODE == PBSIM_RNG_PHILOX) {
    if (!slow) {
      qshmm_simulate_fast(T, A.keys, (uint32_t)(A.B.first_read + 1u + r), pass, wlen, sink.ev, sink.ck, sink.cap, res);
    } else {
      PhiloxDrawQ d;
      d.ph.k0 = A.rng.seed;
      d.ph.k1 = A.G.seq_num;
      d.read_id = (uint32_t)(A.B.first_read + 1u + r);
      d.pass = pass;
      qshmm_simulate(T, d, win, slow, wlen, sink, res);
    }
  } else {
    ReplayDraw d;
    replay_setup(d, A.rng, s, pass, A.plan_draws, wlen < A.G.len);
    qshmm_simulate(T, d, win, slow, wlen, sink, res);
    used = d.consumed();
  }
  store_result(A.B, s, res, used);
}

// ----------------------------------------------------------------------------------------------
// K3: errhmm pass 1
// shared memory: [table blob (t2 | emis | emod) | edel (nst+1)*2 rounded | mbarrier]
// ----------------------------------------------------------------------------------------------
template <int RNG_MODE>
__global__ void __launch_bounds__(kErrThreads) k_sim_errhmm(SimArgs A, uint32_t smem_bar_off) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  const AccEntry ae = A.M.acc[acc];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + smem_bar_off);
  const uint32_t edel_bytes = ((ae.nstates + 1u) * 2u + 15u) / 16u * 16u;
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  if (ae.valid && ae.mode != 3u) {
    if (threadIdx.x == 0) {
      mbar_expect_tx(bar, ae.blob_bytes + edel_bytes);
      tma_bulk_g2s(smem, A.M.blob + ae.blob_off, ae.blob_bytes, bar);
      tma_bulk_g2s(smem + ae.blob_bytes, A.M.er_bias + ae.bias_off, edel_bytes, bar);
    }
    mbar_wait(bar, 0);
  }
  const uint32_t k = lo + threadIdx.x;
  if (k >= hi) return;
  const uint32_t s = A.B.order[k];
  const uint32_t r = s / A.M.pass_num, pass = s % A.M.pass_num;
  const uint32_t meta = A.B.plan_meta[r];
  const uint32_t wlen = A.B.plan_wlen[r];
  if (meta & (1u << 10)) {
    SubreadResult z = {};
    z.overflow = 2;
    store_result(A.B, s, z, 0);
    return;
  }
  ErView T;
  uint32_t t2o, emo, emodo;
  er_blob_bytes(ae.nstates, &t2o, &emo, &emodo);
  T.t2 = reinterpret_cast<const uint16_t *>(smem + t2o);
  T.emis = smem + emo;
  T.emod = reinterpret_cast<const uint16_t *>(smem + emodo);
  T.edel = reinterpret_cast<const uint16_t *>(smem + ae.blob_bytes);
  T.edel_hp = A.M.er_bias + ae.bias_off + (ae.nstates + 1u);
  T.init_mod = ae.init_mod;
  T.mode = ae.mode;
  T.rate_mag = ae.rate_mag;
  WindowRef win;
  win.ascii = A.G.ascii;
  win.hp4 = A.G.hp4;
  win.offset = A.B.plan_off[r];
  win.wlen = wlen;
  win.minus = (meta >> 8) & 1u;
  const bool slow = (meta >> 9) & 1u;
  ErSink sink;
  sink.init(A.ev + A.B.ev_off[s], A.ck + A.B.ck_off[s], A.B.cap[s]);
  SubreadResult res;
  uint32_t used = 0;
  if (RNG_MODE == PBSIM_RNG_PHILOX) {
    PhiloxDraw d;
    d.ph.k0 = A.rng.seed;
    d.ph.k1 = A.G.seq_num;
    d.read_id = (uint32_t)(A.B.first_read + 1u + r);
    d.pass = pass;
    errhmm_simulate(T, d, win, slow, wlen, sink, res);
  } else {
    ReplayDraw d;
    replay_setup(d, A.rng, s, pass, A.plan_draws, wlen < A.G.len);
    errhmm_simulate(T, d, win, slow, wlen, sink, res);
    used = d.consumed();
  }
  store_result(A.B, s, res, used);
}

// ----------------------------------------------------------------------------------------------
// --method sample (simulate_by_sample, pbsim.cpp:1694-1949; schedule: sample_plan.hpp)
// The reads of a batch are the copies of GROUPS (pool entry, pool pass) in read order; the copies of a group are
// a chain (copy i+1 is as long as copy i's read), so ONE thread simulates a group: it plans copy 0 from the pool
// entry's length, runs sample_simulate, plans copy 1 from the read's length, and so on.  Groups run in parallel,
// scheduled longest-first like the sequential pass-1 bins (bin 0; copies > 0 carry the out-of-range bin).
//
// Speculation (option "sample_spec", default on): with the usual error mix (more insertions than deletions) a read
// uses up its quality string before its window, so every copy is as long as the pool entry and the chain is
// trivial.  The engine therefore first simulates EVERY copy in its own thread assuming the entry's length
// (critical path: one read instead of all copies of the longest entry), k_sample_redo then finds, per group, the
// first copy whose predecessor came out shorter than assumed, and only those tails are redone as chains that start
// from the predecessor's read length.  The result is the chain's, by construction.
// ----------------------------------------------------------------------------------------------
struct DevicePool {
  const uint8_t *quals;    // quality strings of the filtered sample reads, concatenated (fp_filtered, :1214-1275)
  const uint64_t *start;   // [n+1]
  uint32_t n;
};

struct SampleBatch {
  const uint32_t *g_entry;  // [n_groups] pool entry
  const uint32_t *g_first;  // [n_groups+1] first read of the group inside the batch
  uint32_t n_groups;
  uint32_t skip_first;      // replay: read 0 of the batch is preceded by the pool-pass draw (:1734)
};

// seg_min_len != 0 (speculative pass, PHILOX draws, --hp-del-bias 1): reads of at least that many positions are planned
// here completely (offset, strand: what k_sim_sample does for the others) and cut into segments of
// PB_TILE positions for the error pass (k_sim_seg<true>: the qualities come from the pool entry) and k_find_end.
__global__ void k_plan_sample(DeviceGenome G, DevicePool Pl, SampleBatch SB, Batch B, uint32_t cap_num, uint32_t cap_den,
                              uint32_t spec, uint32_t seed, uint32_t uniform_bias, uint32_t seg_min_len) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= B.n_reads) return;
  uint32_t lo = 0, hi = SB.n_groups;  // g_first[lo] <= r < g_first[hi]
  while (hi - lo > 1u) {
    const uint32_t mid = (lo + hi) >> 1;
    if (SB.g_first[mid] <= r) lo = mid;
    else hi = mid;
  }
  const uint32_t copy = r - SB.g_first[lo], num = SB.g_first[lo + 1] - SB.g_first[lo];
  const uint32_t j = SB.g_entry[lo];
  const uint32_t entry_len = (uint32_t)(Pl.start[j + 1] - Pl.start[j]);
  uint32_t len0 = entry_len;
  if (len0 > G.len) len0 = G.len;
  B.plan_tr[r] = j;
  B.plan_off[r] = 0;
  B.plan_wlen[r] = len0;   // upper bound; the group's thread stores the planned window of every copy
  B.plan_raw[r] = spec ? 1u : num;  // copies the thread scheduled for this read simulates (chain: copy 0 walks them all)
  B.plan_meta[r] = 0;
  bool segmented = false;
  if (seg_min_len != 0u && spec && len0 >= seg_min_len && uniform_bias) {
    const uint32_t read_id = (uint32_t)(B.first_read + 1u + r);
    PhiloxDrawQ pd;
    pd.ph.k0 = seed;
    pd.ph.k1 = G.seq_num;
    pd.read_id = read_id;
    pd.pass = 0;
    pd.plan_begin();
    const uint32_t offset = entry_len >= G.len ? 0u : pd.plan_off(G.len - len0 + 1u);  // :1758-1763
    // a window that touches an exceptional block (a non-ACGT base, a homopolymer of 11 or more) is segmented too, as
    // for qshmm: k_find_end repairs its deletion runs with the exact reference offset, pass 2 takes the generic path
    const bool slow = range_exceptional(G.xm, offset, offset + len0 - 1u);
    segmented = true;
    const uint32_t minus = (read_id & 1u) ? 0u : 1u;  // :1768-1774
    B.plan_off[r] = offset;
    B.plan_meta[r] = (minus << 8) | ((slow ? 1u : 0u) << 9) | (1u << 11);
  }
  uint64_t cap = (uint64_t)len0 * cap_num / cap_den + 2048u;
  const uint32_t nseg = segmented ? (len0 + PB_TILE - 1u) / PB_TILE : 0u;
  if (segmented) cap = (uint64_t)nseg * PB_SEG_STRIDE + 64u;
  cap = (cap + 7u) / 8u * 8u;
  uint64_t work = spec ? (uint64_t)len0 : (uint64_t)len0 * num / 16u;
  if (work > 0xFFFFFu) work = 0xFFFFFu;
  // segmented reads carry the out-of-range bin: the sequential schedule skips them (as it skips copies > 0 of a chain)
  B.key_in[r] = (!segmented && (copy == 0u || spec)) ? (0xFFFFFu - (uint32_t)work) : ((uint32_t)kBins << 20);
  B.idx_in[r] = r;
  B.cap[r] = (uint32_t)cap;
  B.ck_cap[r] = segmented ? nseg + 2u : (uint32_t)(cap / PB_TILE) + 2u;
  B.nseg[r] = nseg;
  B.nchunk[r] = 0;
  B.grp_copy[r] = copy;
  B.grp_num[r] = num;
}

// after the speculative pass: read r heads a chain to redo iff its predecessor's read is not as long as r assumed
// and every earlier copy of the group assumed right; everything else leaves the schedule
__global__ void k_sample_redo(Batch B, unsigned long long *n_redo) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= B.n_reads) return;
  const uint32_t copy = B.grp_copy[r], num = B.grp_num[r];
  bool head = copy > 0u && B.rlen[r - 1u] != B.plan_wlen[r];
  for (uint32_t k = 1; head && k < copy; ++k)
    if (B.rlen[r - copy + k - 1u] != B.plan_wlen[r - copy + k]) head = false;
  uint32_t key = (uint32_t)kBins << 20;
  if (head) {
    uint64_t work = (uint64_t)B.plan_wlen[r] * (num - copy) / 16u;
    if (work > 0xFFFFFu) work = 0xFFFFFu;
    key = 0xFFFFFu - (uint32_t)work;
    B.plan_raw[r] = num - copy;
    atomicAdd(n_redo, 1ull);
  }
  B.key_in[r] = key;
  B.idx_in[r] = r;
}

// shared memory: the per-quality tables (thr | qc_prob | thr32 | fast)
constexpr uint32_t kSampleSmemBytes = kQsTabBytes;

template <int RNG_MODE>
__global__ void __launch_bounds__(kSimThreads) k_sim_sample(SimArgs A, DevicePool Pl, SampleBatch SB,
                                                            uint32_t from_prev /* redo pass: chains start at any copy */) {
  __shared__ __align__(16) uint8_t smem[kSampleSmemBytes];
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  {
    uint32_t *d = reinterpret_cast<uint32_t *>(smem);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(A.M.qs_tabs);
    for (uint32_t i = threadIdx.x; i < kQsTabBytes / 4u; i += blockDim.x) d[i] = src[i];
  }
  __syncthreads();
  const uint32_t k = lo + threadIdx.x;
  if (k >= hi) return;
  const uint32_t r0 = A.B.order[k];
  const uint32_t num = A.B.plan_raw[r0];
  const uint32_t j = A.B.plan_tr[r0];
  const uint8_t *quals = Pl.quals + Pl.start[j];
  QsView T;
  T.t2 = nullptr;
  T.emis = nullptr;
  T.freq = nullptr;
  T.has_model = 0;
  T.init_mod = 1;
  T.freq_mod = 1;
  T.thr = reinterpret_cast<const QsThr *>(smem + kQsTabThr);
  T.thr_hp = A.M.qs_thr_hp;
  T.qc_prob = reinterpret_cast<const double *>(smem + kQsTabProb);
  T.thr32 = reinterpret_cast<const QsThr *>(smem + kQsTabThr32);
  T.thr_hp32 = A.M.qs_thr_hp32;
  T.fast = reinterpret_cast<const QsFast *>(smem + kQsTabFast);
  uint32_t len = (uint32_t)(Pl.start[j + 1] - Pl.start[j]);
  if (from_prev) len = A.B.rlen[r0 - 1u];  // the buffer was cut where the previous copy's read ended
  for (uint32_t i = 0; i < num; ++i) {
    const uint32_t r = r0 + i;
    const uint32_t read_id = (uint32_t)(A.B.first_read + 1u + r);
    PhiloxDrawQ pd;
    ReplayDraw rd;
    uint32_t offset = 0;
    if (RNG_MODE == PBSIM_RNG_PHILOX) {
      pd.ph.k0 = A.rng.seed;
      pd.ph.k1 = A.G.seq_num;
      pd.read_id = read_id;
      pd.pass = 0;
      pd.plan_begin();
      if (len >= A.G.len) len = A.G.len;                    // :1758-1763
      else offset = pd.plan_off(A.G.len - len + 1u);
    } else {
      rd.log = A.rng.draws - A.rng.draws_base;
      rd.start = A.rng.starts[r];
      rd.cur = rd.start + ((r == 0u && SB.skip_first) ? 1 : 0);
      rd.end = A.rng.draws_end;
      if (len >= A.G.len) len = A.G.len;
      else offset = rd.plan_off(A.G.len - len + 1u);
    }
    const uint32_t minus = (read_id & 1u) ? 0u : 1u;       // :1768-1774
    bool slow = !A.M.uniform_bias;
    if (!slow && len > 0u) slow = range_exceptional(A.G.xm, offset, offset + len - 1u);
    A.B.plan_off[r] = offset;
    A.B.plan_wlen[r] = len;
    A.B.plan_meta[r] = (minus << 8) | ((slow ? 1u : 0u) << 9);
    WindowRef win;
    win.ascii = A.G.ascii;
    win.hp4 = A.G.hp4;
    win.offset = offset;
    win.wlen = len;
    win.minus = minus;
    QsSink sink;
    sink.init(reinterpret_cast<uint16_t *>(A.ev) + A.B.ev_off[r], A.ck + A.B.ck_off[r], A.B.cap[r]);
    SubreadResult res;
    uint32_t used = 0;
    if (RNG_MODE == PBSIM_RNG_PHILOX) {
      sample_simulate(T, pd, win, slow, len, quals, sink, res);
    } else {
      sample_simulate(T, rd, win, slow, len, quals, sink, res);
      used = rd.consumed();
    }
    store_result(A.B, r, res, used);
    len = res.rlen;  // mut.qc was cut where the read ended (:1835): the next copy is this long (:1756)
  }
}

}  // namespace pb
