// Segment-parallel pass 1 (PHILOX mode).  See sim_core.cuh "qshmm SEGMENT-PARALLEL pass 1".
//
// Long reads are cut into segments of PB_TILE read positions (qshmm) / alignment columns (errhmm), so the work
// units are the same size whatever the read lengths are (1 kb or 1 Mb), which removes the sequential critical
// path a whole-read-per-thread schedule has.  qshmm splits the work by what is sequential and what is not:
//   k_seg_fill    : (sub-read, k) list of all segments of the batch + accuracy sort key
//   k_qs_pass1    : model accuracies.  One thread per chunk of segments: exact entry state by backward coupling,
//                   then the HMM chain + emission walk and, position by position, the error draw, choices and
//                   deletion run -> the events and the segments' totals
//   k_sim_seg     : accuracies without a model (and --method sample).  One WARP per segment, consecutive lanes on
//                   consecutive positions: quality, error draw, choices, deletion run -> the event (coalesced)
//   k_find_end    : one warp per segmented sub-read: prefix over its segments, deletion-run repairs, clip at the
//                   window end, tile checkpoints, totals
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sim_kernels.cuh"

namespace pb {

struct SegBatch {
  uint32_t n_seg_total;
  const uint64_t *seg_off;   // [n_sub + 1] exclusive scan of segments per sub-read (0 for sequential sub-reads)
  uint32_t *seg_sub;         // [n_seg_total] sub-read of a segment
  uint32_t *seg_key_in;      // [n_seg_total] accuracy << 21 (same bin arithmetic as the sequential schedule)
  uint32_t *seg_key_out;
  uint32_t *seg_id_in;
  uint32_t *seg_order;       // segments sorted by accuracy
  SegResult *seg_res;        // [n_seg_total] indexed by segment id
  uint32_t *seg_state;       // [n_seg_total] chain state in front of a segment (recorded by k_chain_chunk_err)
};

// thread per sub-read: write its segments' descriptors.  skip_chained: the segments of reads whose chain chunks
// simulate them (qshmm model accuracies, k_qs_pass1) get the out-of-range bin kBins, so k_sim_seg skips them
__global__ void k_seg_fill(Batch B, SegBatch S, uint32_t pass_num, uint32_t skip_chained) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= B.n_sub) return;
  const uint64_t lo = S.seg_off[s], hi = S.seg_off[s + 1];
  if (hi == lo) return;
  const uint32_t meta = B.plan_meta[s / pass_num];
  const uint32_t acc = meta & 0xFFu;
  const bool skip = skip_chained != 0u && B.nchunk[s] != 0u;
  for (uint64_t i = lo; i < hi; ++i) {
    S.seg_sub[i] = s;
    S.seg_key_in[i] = skip ? ((uint32_t)kBins << 20) : acc << 21;
    S.seg_id_in[i] = (uint32_t)i;
  }
}

// ---- chain chunks: the threads that recover the HMM state in front of every segment -------------------------------
struct ChunkBatch {
  uint32_t n_chunks, per_chunk;   // per_chunk: segments walked by one chunk (reads of sticky chains: all of them)
  uint32_t qs;                    // 1: qshmm (k_qs_pass1 walks every segment)
  const uint64_t *chunk_off;      // [n_sub + 1] exclusive scan of Batch::nchunk
  uint32_t *sub, *key_in, *key_out, *id_in, *order;
};

__global__ void k_chunk_fill(Batch B, ChunkBatch C, uint32_t pass_num) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= B.n_sub) return;
  const uint64_t lo = C.chunk_off[s], hi = C.chunk_off[s + 1];
  if (hi == lo) return;
  const uint32_t acc = B.plan_meta[s / pass_num] & 0xFFu;
  const uint32_t nseg = B.nseg[s];
  const uint32_t per = (hi - lo == 1u) ? nseg : C.per_chunk;
  for (uint64_t i = lo; i < hi; ++i) {
    // longest walk first inside an accuracy (the same key layout as the sequential schedule)
    // errhmm records the state in front of segments k_from+1 .. k_to (nobody needs the one behind the last
    // segment); qshmm's k_qs_pass1 walks every segment
    const bool qs = C.qs != 0u;
    const uint32_t k_from = (uint32_t)(i - lo) * per, k_to = min(k_from + per, qs ? nseg : nseg - 1u);
    const uint32_t work = k_to - k_from + (k_from > 0u ? 1u : 0u);
    C.sub[i] = s;
    C.key_in[i] = (acc << 21) | (0xFFFFFu - min(work, 0xFFFFFu));
    C.id_in[i] = (uint32_t)i;
  }
}

struct SegArgs {
  PhiloxKeys keys;
  DeviceModel M;
  DeviceGenome G;
  const uint8_t *bias_one;
  Batch B;
  SegBatch S;
  const uint32_t *cta_order, *cta_first, *bin_lo, *bin_hi;
  uint8_t *ev;
  // --method sample: the pool of quality strings (the qualities of a read's positions are its pool entry's bytes)
  const uint8_t *pool_q;
  const uint64_t *pool_start;
};

// The qshmm segments without chain chunks (accuracies without a model, --method sample): one WARP per segment, lane l
// of iteration i on positions 128 i + 4 l .. + 3.  The qualities come from the freq2qc table or the pool entry; the
// events are written with 8-byte stores, consecutive lanes on consecutive addresses.
// A CTA serves kSimThreads segments of one accuracy (the schedule of the other pass-1 kernels), warp w the
// segments lo + w, lo + w + 4, ...
constexpr int kSegWarps = kSimThreads / 32;
// threads of a chain-chunk CTA (they share one accuracy's tables, 30 KB: 7 CTAs per SM with the largest shared-memory
// carve-out).  Measured on the quality pass alone: 256-thread CTAs (48 warps per SM) were 15 % slower (c3 and c1,
// chunks of 8 segments), 512-thread CTAs likewise with chunks of 32 — more warps only queue up behind the shared-memory
// pipe.
#ifndef PB_CHAIN_THREADS
#define PB_CHAIN_THREADS 128
#endif
constexpr int kChainThreads = PB_CHAIN_THREADS;

// SAMPLE (--method sample, speculative pass): the quality of position p is byte p of the read's pool entry
// (simulate_by_sample, :1775-1833); positions behind the entry's end are filled with quality 0 and dropped by k_find_end.
template <bool SAMPLE>
__global__ void __launch_bounds__(kSimThreads) k_sim_seg(SegArgs A) {
  __shared__ __align__(16) QsFast s_fast[PBSIM_NQV];
  __shared__ __align__(16) uint8_t s_freq[QsBlobLayout::freq_bytes];
  __shared__ __align__(16) uint8_t s_q[kSegWarps][PB_TILE];  // qualities of a segment that is redone generically
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  AccEntry ae = A.M.acc[SAMPLE ? 0u : acc];
  if (SAMPLE) ae.has_model = 1;  // "the qualities are given": the generic redo of a segment takes them from s_q
  {
    uint32_t *d = reinterpret_cast<uint32_t *>(s_fast);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(A.M.qs_fast);
    for (uint32_t i = threadIdx.x; i < PBSIM_NQV * 4u; i += blockDim.x) d[i] = src[i];
    if (!SAMPLE && !ae.has_model) {
      uint32_t *f = reinterpret_cast<uint32_t *>(s_freq);
      const uint32_t *fs = reinterpret_cast<const uint32_t *>(A.M.blob + ae.blob_off);
      for (uint32_t i = threadIdx.x; i < QsBlobLayout::freq_bytes / 4u; i += blockDim.x) f[i] = fs[i];
    }
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  QsView T;
  T.t2 = nullptr;
  T.emis = nullptr;
  T.freq = s_freq;
  T.has_model = ae.has_model;
  T.init_mod = ae.init_mod;
  T.freq_mod = ae.freq_mod;
  T.thr = nullptr;
  T.thr_hp = nullptr;
  T.qc_prob = nullptr;
  T.thr32 = reinterpret_cast<const QsThr *>(A.M.qs_thr32);  // global: only the rare hp[-1] rule reads it
  T.thr_hp32 = nullptr;
  T.fast = s_fast;
  for (uint32_t i = lo + warp; i < hi; i += kSegWarps) {
    const uint32_t seg = A.S.seg_order[i];
    const uint32_t s = A.S.seg_sub[seg];
    const uint32_t k = seg - (uint32_t)A.S.seg_off[s];
    const uint32_t r = s / A.M.pass_num, pass = s % A.M.pass_num;
    const uint32_t read_id = (uint32_t)(A.B.first_read + 1u + r);
    const uint32_t c1 = pass << 16;
    uint16_t *ev = reinterpret_cast<uint16_t *>(A.ev) + A.B.ev_off[s] + (uint64_t)k * PB_SEG_STRIDE;
    QsLaneTotals t;
    t.nsub = t.nins = t.ndel = t.prob = t.big = 0;
    // the eight 8-byte loads of the lane are independent of everything: all in flight before the first is used
    constexpr uint32_t kIters = PB_TILE / (32u * PB_GROUP);
    uint2 q[kIters];
    if (SAMPLE) {
      const uint8_t *qp = A.pool_q + A.pool_start[A.B.plan_tr[r]];
      const uint32_t len = A.B.plan_wlen[r];
#pragma unroll
      for (uint32_t it = 0; it < kIters; ++it) {
        const uint32_t p = k * PB_TILE + lane * PB_GROUP + it * 32u * PB_GROUP;
        uint32_t b[PB_GROUP];
#pragma unroll
        for (uint32_t u = 0; u < PB_GROUP; ++u) b[u] = p + u < len ? (uint32_t)__ldg(qp + p + u) - 33u : 0u;
        q[it] = make_uint2(b[0] | (b[1] << 16), b[2] | (b[3] << 16));
      }
    }
#pragma unroll
    for (uint32_t it = 0; it < kIters; ++it) {
      const uint32_t j = lane * PB_GROUP + it * 32u * PB_GROUP;
      uint32_t qv[PB_GROUP];
      if (SAMPLE) {
        qv[0] = q[it].x & 0x7Fu; qv[1] = (q[it].x >> 16) & 0x7Fu; qv[2] = q[it].y & 0x7Fu; qv[3] = (q[it].y >> 16) & 0x7Fu;
      } else {
        qs_freq_qualities(T, A.keys, read_id, c1, k * PB_TILE + j, qv);
      }
      uint32_t w0, w1;
      qs_error_lane(s_fast, A.keys, read_id, c1, k * PB_TILE + j, qv, w0, w1, t);
      *reinterpret_cast<uint2 *>(ev + j) = make_uint2(w0, w1);
    }
    const uint32_t big = __any_sync(0xFFFFFFFFu, t.big != 0u) ? 1u : 0u;
    SegResult res;
    if (big) {
      // an entry with >= 15 deletions needs continuation entries: the segment is redone entry by entry
      __syncwarp();
      for (uint32_t j = lane; j < PB_TILE; j += 32u) s_q[warp][j] = (uint8_t)(ev[j] & 0x7Fu);
      __syncwarp();
      if (lane == 0) {
        qshmm_segment_generic(T, A.keys, read_id, pass, k * PB_TILE, k == 0, s_q[warp], ev, res);
        A.S.seg_res[seg] = res;
      }
      __syncwarp();
      continue;
    }
    const uint32_t cnt = __reduce_add_sync(0xFFFFFFFFu, t.nsub | (t.nins << 16));
    uint32_t ndel = __reduce_add_sync(0xFFFFFFFFu, t.ndel);
    const uint32_t plo = __reduce_add_sync(0xFFFFFFFFu, t.prob & 0xFFFFu);
    const uint32_t phi = __reduce_add_sync(0xFFFFFFFFu, t.prob >> 16);
    if (k == 0) {  // leading insertions of the read: the hp[-1] rule (qs_fix_leading)
      __syncwarp();
      if (lane == 0) ndel -= qs_fix_leading(T, A.keys, read_id, c1, ev);
    }
    if (lane == 0) {
      res.n_entries = PB_TILE;
      res.ref_adv = PB_TILE - (cnt >> 16) + ndel;
      res.nsub = cnt & 0xFFFFu;
      res.ndel = ndel;
      res.flags = 0;
      res.pad = 0;
      res.prob = (uint64_t)plo + ((uint64_t)phi << 16);
      A.S.seg_res[seg] = res;
    }
  }
}

// PASS 1 of the qshmm segments of model accuracies: one thread per chain chunk.  Exact state at the chunk's first
// position by backward coupling (init draw at position 0), then qualities and events of every position of the
// chunk's segments in one walk (qshmm_chunk_pass1), which also writes the segments' SegResults.
__global__ void __launch_bounds__(kChainThreads) k_qs_pass1(SegArgs A, ChunkBatch C) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  const AccEntry ae = A.M.acc[acc];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kQsSmemBar);
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, ae.blob_bytes + PBSIM_NQV * 16u);
    tma_bulk_g2s(smem, A.M.blob + ae.blob_off, ae.blob_bytes, bar);
    tma_bulk_g2s(smem + kQsSmemFast, A.M.qs_fast, PBSIM_NQV * 16u, bar);
  }
  mbar_wait(bar, 0);
  const uint32_t i = lo + threadIdx.x;
  if (i >= hi) return;
  const uint32_t id = C.order[i];
  const uint32_t s = C.sub[id];
  const uint32_t c = id - (uint32_t)C.chunk_off[s];
  const uint32_t n_ch = (uint32_t)(C.chunk_off[s + 1] - C.chunk_off[s]);
  const uint32_t r = s / A.M.pass_num, pass = s % A.M.pass_num;
  const uint32_t read_id = (uint32_t)(A.B.first_read + 1u + r);
  const uint32_t nseg = A.B.nseg[s];
  const uint32_t per = n_ch == 1u ? nseg : C.per_chunk;   // a one-chunk read is walked whole
  const uint32_t k_from = c * per, k_to = min(k_from + per, nseg);
  QsView T;
  T.t2 = reinterpret_cast<const uint32_t *>(smem + QsBlobLayout::t2_off);
  T.emis = smem + QsBlobLayout::emis_off;
  T.freq = smem;
  T.has_model = ae.has_model;
  T.init_mod = ae.init_mod;
  T.freq_mod = ae.freq_mod;
  T.thr = nullptr;
  T.thr_hp = nullptr;
  T.qc_prob = nullptr;
  T.thr32 = reinterpret_cast<const QsThr *>(A.M.qs_thr32);  // global: only the rare hp[-1] rule reads it
  T.thr_hp32 = nullptr;
  T.fast = reinterpret_cast<const QsFast *>(smem + kQsSmemFast);
  uint32_t row = 0, mod = ae.init_mod, emod = 1;
  if (k_from > 0u) {
    QsSegAux X;
    X.tmod = smem + QsBlobLayout::tmod_off;
    X.emodv = smem + QsBlobLayout::emodv_off;
    X.reach = ae.reach;
    qshmm_segment_start(T, X, A.keys, read_id, pass, k_from * PB_TILE, ae.seg_ok ? ae.seg_ok : 512u, row, mod, emod);
  }
  // the coupling loops leave the lanes of a warp at different points: reconverge before the walk
  __syncwarp();
  qshmm_chunk_pass1(T, A.keys, read_id, pass, row, mod, k_from, k_to, reinterpret_cast<uint16_t *>(A.ev) + A.B.ev_off[s],
                    A.S.seg_res + A.S.seg_off[s]);
}

// the same for errhmm: chunk 0 walks from column 0 (the init row is drawn until a read base exists, :3853)
__global__ void __launch_bounds__(kErrThreads) k_chain_chunk_err(SegArgs A, ChunkBatch C, uint32_t smem_bar_off) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  const AccEntry ae = A.M.acc[acc];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + smem_bar_off);
  const uint32_t edel_bytes = ((ae.nstates + 1u) * 2u + 15u) / 16u * 16u;
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, ae.blob_bytes + edel_bytes);
    tma_bulk_g2s(smem, A.M.blob + ae.blob_off, ae.blob_bytes, bar);
    tma_bulk_g2s(smem + ae.blob_bytes, A.M.er_bias + ae.bias_off, edel_bytes, bar);
  }
  mbar_wait(bar, 0);
  const uint32_t i = lo + threadIdx.x;
  if (i >= hi) return;
  const uint32_t id = C.order[i];
  const uint32_t s = C.sub[id];
  const uint32_t c = id - (uint32_t)C.chunk_off[s];
  const uint32_t n_ch = (uint32_t)(C.chunk_off[s + 1] - C.chunk_off[s]);
  const uint32_t r = s / A.M.pass_num, pass = s % A.M.pass_num;
  const uint32_t read_id = (uint32_t)(A.B.first_read + 1u + r);
  const uint32_t nseg = A.B.nseg[s];
  const uint32_t per = n_ch == 1u ? nseg : C.per_chunk;
  const uint32_t k_from = c * per, k_to = min(k_from + per, nseg - 1u);
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
  HpProbe hp;
  const uint32_t meta = A.B.plan_meta[r];
  hp.enabled = (meta >> 9) & 1u;
  hp.win.ascii = A.G.ascii;
  hp.win.hp4 = A.G.hp4;
  hp.win.offset = A.B.plan_off[r];
  hp.win.wlen = A.B.plan_wlen[r];
  hp.win.minus = (meta >> 8) & 1u;
  hp.xm = A.G.xm;
  hp.bias_one = A.bias_one;
  uint32_t *rec = A.S.seg_state + A.S.seg_off[s];
  uint32_t state = 0, mod = ae.init_mod;
  bool pzero = true;
  if (k_from == 0u) {  // exact walk from column 0, leading deletions included
    errhmm_state_at(T, A.keys, hp, read_id, pass, k_to * PB_TILE, state, mod, pzero, rec);
    return;
  }
  // tmod[] sits behind emod[] in the blob
  errhmm_segment_start(T, T.emod + (ae.nstates + 1u), ae.reach, A.keys, hp, read_id, pass, k_from * PB_TILE,
                       ae.seg_ok ? ae.seg_ok : 512u, state, mod, pzero);
  __syncwarp();
  if (pzero) {
    // no read base before the chunk (a read that starts with thousands of deletions): walk from column 0; the
    // states in front of this chunk's segments are the only ones written twice, with the same values
    errhmm_state_at(T, A.keys, hp, read_id, pass, k_to * PB_TILE, state, mod, pzero, rec);
    return;
  }
  errhmm_chain_range(T, A.keys, read_id, pass, state, mod, k_from * PB_TILE, k_to * PB_TILE, rec);
}

// One WARP per segmented sub-read.  Same result as qshmm_finish_segmented (sim_core.cuh, the sequential
// statement the CPU harness runs); the exact walk over the entries of a tile is done 32
// entries at a time: a warp scan gives every entry its reference offset; only groups in which the window ends or
// a deletion run meets a flagged block are walked sequentially (by lane 0, with qshmm_walk_tile).
// sample != 0 (--method sample): the read is also over when it is as long as its quality string (= the window length);
// that last position draws no deletion (qshmm_walk_tile, p_left).
__global__ void __launch_bounds__(128) k_find_end(Batch B, SegBatch S, DeviceGenome G, const uint8_t *bias_one,
                                                         uint32_t pass_num, uint8_t *ev, Ckpt *ck, const QsFast *fast,
                                                         uint32_t sample) {
  const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (s >= B.n_sub) return;
  const uint64_t lo = S.seg_off[s], hi = S.seg_off[s + 1];
  if (hi == lo) return;
  const uint32_t r = s / pass_num;
  const uint32_t meta = B.plan_meta[r];
  const uint32_t wlen = B.plan_wlen[r];
  HpProbe hp;
  hp.enabled = (meta >> 9) & 1u;  // window touches an exceptional block: deletion runs may need repairing
  hp.win.ascii = G.ascii;
  hp.win.hp4 = G.hp4;
  hp.win.offset = B.plan_off[r];
  hp.win.wlen = wlen;
  hp.win.minus = (meta >> 8) & 1u;
  hp.xm = G.xm;
  hp.bias_one = bias_one;
  uint16_t *ev_base = reinterpret_cast<uint16_t *>(ev) + B.ev_off[s];
  const SegResult *seg = S.seg_res + lo;
  Ckpt *ckp = ck + B.ck_off[s];
  const uint32_t n_seg = (uint32_t)(hi - lo);
  uint32_t R = 0, P = 0, D = 0, nsub = 0, flags = 0, n_tiles = 0;
  uint64_t prob = 0;
  bool done = false;
  uint32_t k = 0;
  while (k < n_seg && !done) {
    // ---- up to 32 segments at once: lane j looks at segment k + j.  A segment whose reference range neither reaches
    //      the window's end nor touches an exceptional block keeps its own totals: prefix sums over the lanes give
    //      every such segment its checkpoint.  The first segment that needs the exact treatment ends the group.
    {
      const uint32_t kk = k + lane;
      const bool in = kk < n_seg;
      SegResult sr;
      if (in) sr = seg[kk];
      else sr.n_entries = sr.ref_adv = sr.nsub = sr.ndel = sr.flags = sr.pad = 0u, sr.prob = 0ull;
      uint32_t xr = sr.ref_adv, xd = sr.ndel;  // inclusive scans
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t yr = __shfl_up_sync(0xFFFFFFFFu, xr, o), yd = __shfl_up_sync(0xFFFFFFFFu, xd, o);
        if (lane >= (uint32_t)o) xr += yr, xd += yd;
      }
      // (a group that would overflow 32 bits holds a segment that reaches the window's end: 64-bit test)
      const uint64_t Rk64 = (uint64_t)R + xr - sr.ref_adv;
      const uint32_t Rk = (uint32_t)Rk64, Dk = D + xd - sr.ndel;
      bool simple = in && Rk64 + sr.ref_adv < wlen;
      if (sample && (uint64_t)(kk + 1u) * PB_TILE >= wlen) simple = false;  // holds the read's last position
      if (simple && hp.enabled) {
        const uint32_t lo_w = Rk == 0u ? 0u : Rk - 1u, hi_w = Rk + sr.ref_adv;
        const uint32_t ga = hp.win.gidx(lo_w), gb = hp.win.gidx(hi_w);
        simple = !range_exceptional(G.xm, min(ga, gb), max(ga, gb));
      }
      const uint32_t bad = __ballot_sync(0xFFFFFFFFu, !simple);
      const uint32_t cnt = bad ? (uint32_t)__ffs((int)bad) - 1u : 32u;
      if (cnt > 0u) {
        const bool mine = lane < cnt;
        uint32_t f = mine ? sr.flags : 0u;
        if (mine && kk >= 1u && Rk == 0u) f |= 8u;
        flags |= __reduce_or_sync(0xFFFFFFFFu, f);
        if (mine) {
          Ckpt c; c.col = P + lane * PB_TILE + Dk; c.ref = Rk; c.read = P + lane * PB_TILE; c.pad = sr.n_entries;
          ckp[kk] = c;
        }
        R += __shfl_sync(0xFFFFFFFFu, xr, cnt - 1u);
        D += __shfl_sync(0xFFFFFFFFu, xd, cnt - 1u);
        nsub += __reduce_add_sync(0xFFFFFFFFu, mine ? sr.nsub : 0u);
        // prob < 2^36 per segment: 24 + 12 bits
        prob += (uint64_t)__reduce_add_sync(0xFFFFFFFFu, mine ? (uint32_t)(sr.prob & 0xFFFFFFu) : 0u) +
                ((uint64_t)__reduce_add_sync(0xFFFFFFFFu, mine ? (uint32_t)(sr.prob >> 24) : 0u) << 24);
        P += cnt * PB_TILE;
        k += cnt;
        continue;
      }
    }
    // ---- segment k: the window may end in it, or a deletion run may need a repair
    flags |= seg[k].flags;
    if (k >= 1u && R == 0u) flags |= 8u;
    uint16_t *e = ev_base + (uint64_t)k * PB_SEG_STRIDE;
    const uint32_t n = seg[k].n_entries;
    const uint32_t R_tile = R, P_tile = P, D_tile = D;
    uint32_t n_incl = n, blocked = 0;
    bool ended = false;
    for (uint32_t i = 0; i < n && !ended; i += 32u) {
      const uint32_t idx = i + lane;
      const bool valid = idx < n;
      const uint32_t v = valid ? (uint32_t)e[idx] : (uint32_t)PB_QS_PAD;
      const uint32_t kind = (v >> 7) & 3u;
      const bool cont = kind == 3u;
      const uint32_t part = cont ? ((v & 0x7Fu) | ((v >> 9) << 7)) : (v >> 12);
      const uint32_t a = (!cont && kind != PB_KIND_INS) ? 1u : 0u;
      uint32_t x = a + part;  // inclusive scan of reference advances
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= (uint32_t)o) x += y;
      }
      const uint32_t total = __shfl_sync(0xFFFFFFFFu, x, 31);
      const uint32_t Rb = R + x - (a + part);  // reference offset in front of this entry
      // does any deletion of this entry follow a base of a flagged block?  (window indices Rb+a-1 .. Rb+a+part-2)
      bool touch = false;
      if (hp.enabled && part != 0u) {
        const uint32_t w0 = Rb + a, w1 = Rb + a + part - 1u;  // bases whose predecessor matters: w0-1 .. w1-1
        const uint32_t lo_w = w0 == 0u ? 0u : w0 - 1u, hi_w = min(w1 == 0u ? 0u : w1 - 1u, wlen - 1u);
        const uint32_t g0 = hp.win.minus ? hp.win.gidx(hi_w) : hp.win.gidx(lo_w);
        const uint32_t g1 = hp.win.minus ? hp.win.gidx(lo_w) : hp.win.gidx(hi_w);
        touch = range_exceptional(G.xm, g0, g1);
      }
      const uint32_t mb = __ballot_sync(0xFFFFFFFFu, valid && !cont);
      const bool need = __any_sync(0xFFFFFFFFu, touch) || (R + total >= wlen) || blocked != 0u ||
                        (sample && P + (uint32_t)__popc(mb) >= wlen);
      if (!need) {
        const uint32_t ms = __ballot_sync(0xFFFFFFFFu, valid && kind == PB_KIND_SUB);
        uint32_t dsum = part;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dsum += __shfl_down_sync(0xFFFFFFFFu, dsum, o);
        dsum = __shfl_sync(0xFFFFFFFFu, dsum, 0);
        P += __popc(mb);
        nsub += __popc(ms);
        D += dsum;
        R += total;
      } else {
        // exact sequential walk of these (at most 32) entries
        uint32_t res[6];
        if (lane == 0) {
          const TileWalk t = qshmm_walk_tile(e + i, min(32u, n - i), R, wlen, fast, hp, &blocked,
                                             sample ? wlen - P : 0xFFFFFFFFu);
          res[0] = t.n_entries; res[1] = t.positions; res[2] = t.ref_adv; res[3] = t.nsub; res[4] = t.ndel;
          res[5] = t.ended | (blocked << 1);
        }
#pragma unroll
        for (int q = 0; q < 6; ++q) res[q] = __shfl_sync(0xFFFFFFFFu, res[q], 0);
        __syncwarp();
        P += res[1]; R += res[2]; nsub += res[3]; D += res[4];
        blocked = res[5] >> 1;
        if (res[5] & 1u) {
          ended = true;
          n_incl = i + res[0];
        }
      }
    }
    if (lane == 0) {
      Ckpt c; c.col = P_tile + D_tile; c.ref = R_tile; c.read = P_tile; c.pad = n_incl;
      ckp[k] = c;
    }
    if (ended) {
      // fixed-point sum of the error probabilities of the partial tile (order independent)
      uint32_t pp = 0;  // <= 32 positions per lane, each < 2^26
      for (uint32_t i = lane; i < n_incl; i += 32u) {
        const uint32_t v = e[i];
        if (((v >> 7) & 3u) != 3u) pp += fast[v & 0x7Fu].prob;
      }
      prob += (uint64_t)__reduce_add_sync(0xFFFFFFFFu, pp & 0xFFFFu) + ((uint64_t)__reduce_add_sync(0xFFFFFFFFu, pp >> 16) << 16);
      n_tiles = k + 1u;
      done = true;
    } else {
      prob += seg[k].prob;
    }
    ++k;
  }
  if (!done) flags |= 4u;
  if (lane == 0) {
    B.nent[s] = n_tiles;
    B.rlen[s] = P;
    B.ncol[s] = P + D;
    B.nsub[s] = nsub;
    B.nins[s] = P + D - R;
    B.ndel[s] = D;
    B.flags[s] = flags ? (4u | (flags << 8)) : 0u;
    B.draws_used[s] = 0;
    B.accuracy[s] = 1.0 - (((double)prob / (double)(1u << PB_PROB_SHIFT)) / (double)P);
  }
}

// ---------------------------------------------------------------------------------------------
// errhmm
// ---------------------------------------------------------------------------------------------
// shared memory: [table blob (t2 | emis | emod,tmod) | edel rounded | mbarrier]  (same layout as k_sim_errhmm)
__global__ void __launch_bounds__(kErrThreads) k_sim_seg_err(SegArgs A, uint32_t smem_bar_off) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t acc, lo, hi;
  if (!cta_assignment(A.cta_order, A.cta_first, A.bin_lo, A.bin_hi, &acc, &lo, &hi)) return;
  const AccEntry ae = A.M.acc[acc];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + smem_bar_off);
  const uint32_t edel_bytes = ((ae.nstates + 1u) * 2u + 15u) / 16u * 16u;
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, ae.blob_bytes + edel_bytes);
    tma_bulk_g2s(smem, A.M.blob + ae.blob_off, ae.blob_bytes, bar);
    tma_bulk_g2s(smem + ae.blob_bytes, A.M.er_bias + ae.bias_off, edel_bytes, bar);
  }
  mbar_wait(bar, 0);
  const uint32_t i = lo + threadIdx.x;
  if (i >= hi) return;
  const uint32_t seg = A.S.seg_order[i];
  const uint32_t s = A.S.seg_sub[seg];
  const uint32_t k = seg - (uint32_t)A.S.seg_off[s];
  const uint32_t r = s / A.M.pass_num, pass = s % A.M.pass_num;
  const uint32_t read_id = (uint32_t)(A.B.first_read + 1u + r);
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
  uint32_t state = 0, mod = ae.init_mod;
  bool pzero = true;
  bool ok = true;
  if (k > 0) {  // recorded by k_chain_chunk_err
    const uint32_t t = A.S.seg_state[seg];
    state = t & 63u;
    mod = (t >> 6) & 0x3FFu;
    pzero = (t >> 31) != 0u;
  }
  SegResult res;
  if (!ok) {
    res.n_entries = 0; res.ref_adv = 0; res.nsub = 0; res.ndel = 0; res.flags = 2u; res.prob = 0.0;
    A.S.seg_res[seg] = res;
    return;
  }
  errhmm_simulate_segment(T, A.keys, read_id, pass, k * PB_TILE, pzero, state, mod, A.ev + A.B.ev_off[s] + (uint64_t)k * PB_TILE,
                          res);
  A.S.seg_res[seg] = res;
}

// One warp per segmented errhmm sub-read: same result as errhmm_finish_segmented (sim_core.cuh)
__global__ void __launch_bounds__(128) k_find_end_err(Batch B, SegBatch S, DeviceGenome G, PhiloxKeys K,
                                                      const uint8_t *bias_one, uint32_t pass_num, uint8_t *ev, Ckpt *ck) {
  const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (s >= B.n_sub) return;
  const uint64_t lo = S.seg_off[s], hi = S.seg_off[s + 1];
  if (hi == lo) return;
  const uint32_t r = s / pass_num, pass = s % pass_num;
  const uint32_t meta = B.plan_meta[r];
  const uint32_t wlen = B.plan_wlen[r];
  const uint32_t read_id = (uint32_t)(B.first_read + 1u + r);
  HpProbe hp;
  hp.enabled = (meta >> 9) & 1u;
  hp.win.ascii = G.ascii;
  hp.win.hp4 = G.hp4;
  hp.win.offset = B.plan_off[r];
  hp.win.wlen = wlen;
  hp.win.minus = (meta >> 8) & 1u;
  hp.xm = G.xm;
  hp.bias_one = bias_one;
  uint8_t *ev_base = ev + B.ev_off[s];
  const SegResult *seg = S.seg_res + lo;
  Ckpt *ckp = ck + B.ck_off[s];
  const uint32_t n_seg = (uint32_t)(hi - lo);
  const uint32_t lt = (1u << lane) - 1u;
  uint32_t R = 0, P = 0, C = 0, nsub = 0, nins = 0, ndel = 0, flags = 0;
  bool done = false;
  for (uint32_t k = 0; k < n_seg && !done; ++k) {
    flags |= seg[k].flags;
    if (lane == 0) {
      Ckpt c; c.col = C; c.ref = R; c.read = P; c.pad = PB_TILE;
      ckp[k] = c;
    }
    bool seg_touch = false;  // errhmm tests the bias of the CURRENT reference base: window bases R .. R+ref_adv
    if (hp.enabled && (uint64_t)R + seg[k].ref_adv < wlen) {
      const uint32_t ga = hp.win.gidx(R), gb = hp.win.gidx(R + seg[k].ref_adv);
      seg_touch = range_exceptional(G.xm, min(ga, gb), max(ga, gb));
    }
    if (!seg_touch && (uint64_t)R + seg[k].ref_adv < wlen) {
      P += PB_TILE - seg[k].ndel; R += seg[k].ref_adv; nsub += seg[k].nsub; nins += (uint32_t)seg[k].prob;
      ndel += seg[k].ndel; C += PB_TILE;
      continue;
    }
    uint8_t *e = ev_base + (uint64_t)k * PB_TILE;
    for (uint32_t i = 0; i < PB_TILE && !done; i += 32u) {
      const uint32_t v = e[i + lane];
      const uint32_t kind = v & 3u;
      const bool adv = kind != PB_KIND_INS;
      const uint32_t m_adv = __ballot_sync(0xFFFFFFFFu, adv);
      const uint32_t Rb = R + __popc(m_adv & lt);
      const uint32_t total = __popc(m_adv);
      bool touch = false;
      if (hp.enabled && (v & 0x80u) && Rb < wlen) {
        const uint32_t g = hp.win.gidx(Rb);
        touch = range_exceptional(G.xm, g, g);
      }
      const bool need = __any_sync(0xFFFFFFFFu, touch) || (R + total >= wlen);
      if (!need) {
        const uint32_t m_del = __ballot_sync(0xFFFFFFFFu, kind == PB_KIND_DEL);
        const uint32_t m_sub = __ballot_sync(0xFFFFFFFFu, kind == PB_KIND_SUB);
        P += 32u - __popc(m_del);
        R += total;
        nsub += __popc(m_sub);
        nins += 32u - total;
        ndel += __popc(m_del);
        C += 32u;
      } else {
        uint32_t res[8];
        if (lane == 0) {
          const ErTileWalk t = errhmm_walk_tile(e + i, 32u, R, P, wlen, hp, K, read_id, pass, k * PB_TILE + i);
          res[0] = t.n_entries; res[1] = t.positions; res[2] = t.ref_adv; res[3] = t.nsub; res[4] = t.nins;
          res[5] = t.ndel; res[6] = t.ended; res[7] = t.early_repair;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) res[q] = __shfl_sync(0xFFFFFFFFu, res[q], 0);
        __syncwarp();
        P += res[1]; R += res[2]; nsub += res[3]; nins += res[4]; ndel += res[5]; C += res[0];
        if (res[7]) flags |= 8u;
        if (res[6]) done = true;
      }
    }
  }
  if (!done) flags |= 4u;
  if (lane == 0) {
    B.nent[s] = C;  // errhmm tiles are contiguous: total number of columns
    B.rlen[s] = P;
    B.ncol[s] = C;
    B.nsub[s] = nsub;
    B.nins[s] = nins;
    B.ndel[s] = ndel;
    B.flags[s] = flags ? (4u | (flags << 8)) : 0u;
    B.draws_used[s] = 0;
    B.accuracy[s] = 1.0 - ((double)(nsub + nins + ndel) / (double)P);
  }
}

}  // namespace pb
