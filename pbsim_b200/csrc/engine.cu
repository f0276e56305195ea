// libpbsim_cuda — engine orchestration and the C ABI (include/pbsim_cuda.h).
//
// One engine = one GPU.  A simulate_by_* call of the reference (pbsim.cpp:1955 / :3594, the _trans / _templ
// variants :2419, :3055, :4114, :4807, and simulate_by_sample :1694) becomes
//   simulate_begin -> { next_chunk }* -> simulate_end
// and every batch of reads runs, on one stream:
//   K1 k_plan            per-read length / accuracy / offset / strand, segment provisioning  (sim_kernels.cuh)
//      radix sorts       (accuracy, length desc) -> pass-1 schedules                          (CUB, plumbing)
//   K2 k_sim_qshmm | K3 k_sim_errhmm   short reads, replay mode                                (sim_kernels.cuh)
//      k_plan_sample, k_sim_sample, k_sample_redo   --method sample: copies of pool entries     (sim_kernels.cuh)
//      k_sim_seg | k_sim_seg_err, k_find_end[_err]   segment-parallel pass 1 -> event streams (seg_kernels.cuh)
//      quota scan        which read crosses sim.len_quota (pbsim.cpp:2173-2181)               (CUB + k_find_cut)
//   K4 k_sizes, k_tile_desc, k_emit_rows, k_emit   record placement and text emission          (emit.cuh)
//   K6 k_stats           counters and histograms                                              (emit.cuh)
//      k_gz_hist / k_gz_size / k_gz_encode   option "deflate": gzip members for host delivery (gz_kernels.cuh)
// Host delivery is pipelined: a producer thread generates batch k+1 while batch k streams through pinned staging.
// There is no CPU implementation of any of these steps in this library.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pbsim_cuda.h"
#include "emit.cuh"
#include "gz_kernels.cuh"
#include "k0_genome.cuh"
#include "model_image.hpp"
#include "align.cuh"
#include "sample_plan.hpp"
#include "seg_kernels.cuh"
#include "sim_kernels.cuh"

namespace {

thread_local std::string g_create_error;

// Device memory that grows on demand and is freed with its owner (the engine is deleted on the engine's device).
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { cudaFree(p); }  // no-op for nullptr
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    size_t want = bytes + bytes / 8 + 256;
    void *np = nullptr;
    cudaError_t e = cudaMalloc(&np, want);
    if (e != cudaSuccess) return e;
    if (p) {
      cudaStreamSynchronize(0);
      cudaFree(p);
    }
    p = np;
    cap = want;
    return cudaSuccess;
  }
  template <class T>
  T *as() const { return reinterpret_cast<T *>(p); }
};

struct PinnedBuf {
  void *p = nullptr;
  size_t cap = 0;
  PinnedBuf() = default;
  PinnedBuf(const PinnedBuf &) = delete;
  PinnedBuf &operator=(const PinnedBuf &) = delete;
  ~PinnedBuf() { release(); }
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 4096;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

// quota bookkeeping on the device: first read of the batch whose planned length crosses the quota
__global__ void k_rlen0(const uint32_t *rlen, uint32_t n_reads, uint32_t pass_num, unsigned long long *out) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_reads) out[r] = rlen[(uint64_t)r * pass_num];
}

// ctrl[0] = cut index (first read with len_total + raw_len > quota), n_reads if none
__global__ void k_find_cut(const unsigned long long *prefix, const uint32_t *plan_raw, uint32_t n_reads,
                           long long len_total, long long quota, unsigned long long *ctrl) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  if (len_total + (long long)prefix[r] + (long long)plan_raw[r] > quota) atomicMin(&ctrl[0], (unsigned long long)r);
}

// --method sample tests the quota in front of every read and never clips one (pbsim.cpp:1747, :1753)
__global__ void k_find_cut_sample(const unsigned long long *prefix, uint32_t n_reads, long long len_total, long long quota,
                                  unsigned long long *ctrl) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  if (len_total + (long long)prefix[r] >= quota) atomicMin(&ctrl[0], (unsigned long long)r);
}

// ctrl[1] = emitted bases (pass 0) of the reads before the cut; ctrl[2] = any pass-1 flag
__global__ void k_batch_totals(const unsigned long long *prefix, const uint32_t *rlen, const uint32_t *flags,
                               uint32_t n_reads, uint32_t pass_num, unsigned long long *ctrl) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long cut = ctrl[0];
  if (i == 0) {
    if (cut >= n_reads) ctrl[1] = prefix[n_reads - 1] + rlen[(uint64_t)(n_reads - 1) * pass_num];
    else ctrl[1] = prefix[cut];
  }
  const uint64_t n_sub = (uint64_t)min((unsigned long long)n_reads, cut + 1) * pass_num;
  if (i < n_sub && flags[i]) atomicOr(reinterpret_cast<unsigned int *>(&ctrl[2]), flags[i]);
}

// Control read-backs (a few words per batch) are written by a kernel straight into pinned host memory instead of
// going through cudaMemcpyAsync: a D2H memcpy on the compute stream queues on the same DMA engine as the delivery
// stream's 128 MiB record copies and waits milliseconds behind them, several times per batch.
__global__ void k_peek(const uint32_t *__restrict__ src, uint32_t *__restrict__ host_dst, uint64_t words) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < words) host_dst[i] = src[i];
}

__global__ void k_iota_u32(uint32_t *p, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

__global__ void k_fill_u32(uint32_t *p, uint32_t n, uint32_t v) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

__global__ void k_init_stats(unsigned long long *blk, int64_t cells) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cells) blk[i] = (i == 3) ? (unsigned long long)LLONG_MAX : 0ull;
}

// widen uint32 -> uint64 for the scans
__global__ void k_widen(const uint32_t *in, uint32_t n, unsigned long long *out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}

// replay: number of draws each subread consumed must equal the distance to the next start
__global__ void k_check_replay(const int64_t *starts, const uint32_t *used, const uint32_t *plan_wlen, uint32_t glen,
                               uint32_t n_sub, uint32_t pass_num, int64_t next_start_after,
                               const unsigned long long *ctrl, unsigned int *bad) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_sub) return;
  if ((unsigned long long)(s / pass_num) >= ctrl[0]) return;  // reads at / after the quota cut are re-planned
  const int64_t nxt = (s + 1 < n_sub) ? starts[s + 1] : next_start_after;
  if (nxt < 0) return;  // unknown (last subread of the log)
  // `used` counts from the subread's start, i.e. it already includes the planner's 2 or 3 draws of pass 0
  if (starts[s] + (int64_t)used[s] != nxt) atomicAdd(bad, 1u);
}

}  // namespace

using namespace pb;

struct pbsim_engine {
  int device = 0;
  cudaStream_t st = nullptr, st_copy = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;

  // model
  bool model_set = false;
  pbsim_model model;  // shallow copy: scalar fields only are used after set_model
  ModelImage img;
  std::vector<int32_t> h_prob2len;
  std::vector<uint8_t> h_prob2acc;
  DevBuf d_blob, d_acc, d_prob2len, d_prob2acc, d_qs_tabs, d_qs_thr_hp, d_qs_thr_hp32, d_er_bias;
  std::vector<uint8_t> h_qs_tabs;
  uint32_t er_smem_bar_off = 0;
  EmitParams emitp;

  // sequence
  bool seq_set = false;
  DevBuf d_ascii, d_pk, d_hp4, d_xm, d_hpfreq, d_biasone, d_flag;
  int64_t glen = 0;
  int32_t seq_num = 0;
  double bias[12];
  int64_t hpfreq[12];

  // sequence set (--strategy trans / templ); strategy WGS when a plain sequence is loaded
  int strategy = PBSIM_STRATEGY_WGS;
  int64_t set_n = 0, set_total_reads = 0;
  double set_mean_len = 0;
  int32_t set_rank_max = 0;
  DevBuf d_set_start, d_set_rprefix, d_set_plus, d_set_ids, d_set_idstart, d_set_ssp_ends, d_set_ssp_mod, d_set_first;
  // host copies for the replay read map of simulate_by_errhmm_trans (build_replay_read_map)
  std::vector<uint32_t> h_set_start, h_set_nr;
  std::vector<uint16_t> h_ssp_ends, h_ssp_mod;
  DevBuf d_map_tr, d_map_k;
  bool replay_map = false;

  // --method sample: the pool of quality strings (get_sample_inf's fp_filtered) and the run's schedule
  bool pool_set = false;
  std::vector<int64_t> pool_start;
  DevBuf d_pool_q, d_pool_start, d_groups;
  SampleSchedule sched;
  SampleGroups groups;
  int sample_spec = 1;            // option "sample_spec": simulate all copies at once assuming full-length reads, redo the rest
  bool sample_spec_run = true;    // this run: switched off when most groups had to be redone
  int64_t sample_redo_groups = 0;

  // run
  bool running = false;
  pbsim_run run;
  int64_t next_read = 0;  // reads simulated so far (ids are 1-based: next id = next_read + 1)
  int64_t len_total = 0;
  int64_t reads_done_in_run = 0;
  bool finished = false;
  bool tail_mode = false;
  double mean_rlen_est = 0;
  double table_mean_len = 0;  // mean of the length sampler, for the first batch-size estimate
  uint32_t cap_num = 5, cap_den = 4;  // event-slot capacity = wlen * 5/4 + 2048
  DevBuf d_draws, d_starts;

  // batch arrays
  DevBuf b_read_u32;   // 5 arrays per read (carve_batch)
  DevBuf b_sub_u32;    // 16 arrays per subread
  DevBuf b_sub_u64;    // kU64Slices slices of n_sub + 1 (u64_slice)
  DevBuf b_sub_f64;
  DevBuf d_bins;       // pass-1 CTA schedule of the sub-reads (schedule_ctas)
  DevBuf d_ctrl;       // control words
  DevBuf d_cub_tmp;
  DevBuf d_ev, d_ck, d_lay, d_tile_sub, d_tile_desc;
  DevBuf d_seg, d_seg_bins;       // segment-parallel pass 1: segment lists / results, CTA schedule
  int seg_enabled = 1;            // option "segments"
  int64_t seg_min_len = 2048;     // option "seg_min_len": shorter reads stay on the sequential path
  int64_t seg_batches = 0, seg_fallback_batches = 0;
  // option "chain_chunk": segments walked by one thread of the chain pass; 0 = by method.  Measured on B200 (bench.py,
  // chunks of 2 / 4 / 6 / 8 / 12 / 16 / 24 / 32 / 64 segments): the qshmm quality pass, which walks every position, is
  // fastest with short chunks (more threads hide the dependent shared-memory lookups: c3 108.2 / 107.5 Gbp/s at 4 / 8
  // against 102.0 at 32; c1 88.1 / 89.2 against 85.7); errhmm, whose chunk threads only record states and pay a
  // costlier coupling, with long ones (c2 77.3 at 32 against 74.8 at 8; c5 70.3 against 66.3)
  int64_t chain_chunk = 0;
  uint32_t chain_chunk_eff() const {
    return chain_chunk > 0 ? (uint32_t)chain_chunk : (model.method == PBSIM_METHOD_QSHMM ? 8u : 32u);
  }
  DevBuf d_chunk, d_chunk_bins;
  float seg_extra = 0.0f;         // extra segment headroom (fraction), raised when a batch runs out of segments
  // the records of a batch live in one of two output sets in HBM: with the pipeline on, a producer
  // thread generates batch k+1 into the other set while batch k is handed to the caller
  struct OutSet {
    DevBuf reads, maf;
  } out[2];
  int cur_set = 0;                  // the set run_batch writes
  PinnedBuf h_ctrl, h_acc, h_stats;
  struct BatchItem {
    int rc = 1;                     // 1 = a batch, 0 = the run is finished, < 0 = error (message in err)
    std::string err;
    int set = 0;
    int64_t first_read = 0, n_reads = 0, bases = 0;
    uint64_t reads_bytes = 0, maf_bytes = 0;          // bytes to deliver (gzip members when deflate is on)
    uint64_t reads_text_bytes = 0, maf_text_bytes = 0;
    bool gz = false;
  };
  // option "deflate": host delivery hands out gzip members (gz_kernels.cuh) instead of text
  int deflate = 0;
  int bam = 0;                      // option "bam": multi-pass records are BAM alignment records, not SAM text
  int align = 0;                    // option "align": the second stream holds SAM alignment lines, not MAF blocks
  std::string seq_name;             // RNAME of WGS alignment lines (pbsim_cuda_set_sequence_name; reset by set_sequence)
  DevBuf d_rname, d_aln_rec, d_aln_maf;
  OutSet gz[2];
  DevBuf d_gz_tables, d_gz_hist, d_gz_usize, d_gz_ucrc, d_gz_uoff, d_gz_usel, d_gz_sbits;
  PinnedBuf h_gz;
  double gz_ms = 0, seg_ms = 0, chain_ms = 0;
  cudaEvent_t ev_gz[2] = {nullptr, nullptr}, ev_seg[2] = {nullptr, nullptr}, ev_chain[2] = {nullptr, nullptr};
  int pipeline = 1;                 // option "pipeline": 0 off, 1 host delivery only, 2 always
  int64_t host_batch_bases = (int64_t)1 << 30;  // option: batch size of pipelined host delivery
  int64_t first_batch_div = 1;                  // option: the first batch of a pipelined run can be made this much smaller (measured: no gain)
  bool mode_set = false, mode_to_host = false, pipelined = false;
  std::thread producer;
  std::mutex mu;
  std::condition_variable cv;
  std::deque<BatchItem> queue;
  int free_sets = 2;
  bool stop = false;
  int held_set = -1;                // device delivery: the set the caller's chunk points into
  // host delivery: records are handed out in pieces through two pinned staging buffers per
  // stream (D2H of piece i+1, possibly the first of the next batch, overlaps the caller consuming piece i)
  PinnedBuf h_stage[2][2];          // [stream: 0 reads, 1 maf][slot]
  size_t stage_bytes = (size_t)128 << 20;
  struct Pending {                  // the batch pieces are being issued from
    bool active = false;
    bool gz = false;
    uint64_t text[2] = {0, 0};
    int set = 0;
    uint64_t total[2] = {0, 0}, issued[2] = {0, 0};
    bool first = true;
    int64_t first_read = 0, n_reads = 0, bases = 0;
  } pend;
  struct Piece {                    // the piece in flight into h_stage[*][slot]
    bool valid = false;
    int slot = 0;
    uint64_t bytes[2] = {0, 0};
    bool first = false;
    int64_t first_read = 0, n_reads = 0, bases = 0;
    uint64_t text[2] = {0, 0};      // first piece of a batch: text bytes the batch's members inflate to
    int release_set = -1;           // last piece of its batch: the set is free once this copy is done
  } piece;
  int next_slot = 0;
  std::mutex err_mu;
  cudaEvent_t ev_copy = nullptr, ev_k[4] = {nullptr, nullptr, nullptr, nullptr}, ev_user[2] = {nullptr, nullptr};
  double sim_ms = 0, emit_ms = 0;
  int64_t target_batch_bases = (int64_t)6 << 30;
  Batch B;
  uint64_t *u64_cap_scan = nullptr;
  // last chunk info
  std::vector<int64_t> last_info;

  // stats
  DevBuf d_stats;
  int64_t stats_cells = 0, freq_len_cells = 0;
  double accuracy_total = 0;
  double gen_ms = 0;
  int64_t launches = 0;
};

namespace {

int fail(pbsim_engine *e, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (e) {
    std::lock_guard<std::mutex> lk(e->err_mu);
    e->err = buf;
  } else {
    g_create_error = buf;
  }
  return code;
}

#define CK(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t _e = (call);                                                                              \
    if (_e != cudaSuccess)                                                                                \
      return fail(e, PBSIM_E_CUDA, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__, __LINE__, #call); \
  } while (0)

inline uint32_t nblk(uint64_t n, uint32_t t) { return (uint32_t)((n + t - 1) / t); }

template <class T>
int upload(pbsim_engine *e, DevBuf &d, const T *src, size_t n) {
  CK(d.ensure(std::max<size_t>(n * sizeof(T), 16)));
  if (n) CK(cudaMemcpyAsync(d.p, src, n * sizeof(T), cudaMemcpyHostToDevice, e->st));
  return 0;
}

// device -> pinned host, by a kernel on the engine's stream (see k_peek); host_dst must be pinned memory, both
// pointers 4-byte aligned, bytes a multiple of 4
int peek(pbsim_engine *e, void *host_dst, const void *dev_src, size_t bytes) {
  if (!bytes) return 0;
  const uint64_t words = (bytes + 3) / 4;
  k_peek<<<nblk(words, 256), 256, 0, e->st>>>(reinterpret_cast<const uint32_t *>(dev_src), reinterpret_cast<uint32_t *>(host_dst),
                                              words);
  CK(cudaGetLastError());
  return 0;
}

DeviceModel device_model(const pbsim_engine *e) {
  DeviceModel M;
  M.blob = e->d_blob.as<uint8_t>();
  M.acc = e->d_acc.as<AccEntry>();
  M.prob2len = e->d_prob2len.as<int32_t>();
  M.prob2acc = e->d_prob2acc.as<uint8_t>();
  M.len_rand_value = (uint32_t)e->model.len_rand_value;
  M.acc_rand_value = (uint32_t)e->model.accuracy_rand_value;
  M.len_min = (uint32_t)e->model.len_min;
  M.qs_tabs = e->d_qs_tabs.as<uint8_t>();
  M.qs_thr_hp = e->d_qs_thr_hp.as<uint32_t>();
  M.qs_thr_hp32 = e->d_qs_thr_hp32.as<uint32_t>();
  M.qs_thr32 = reinterpret_cast<const uint32_t *>(M.qs_tabs + kQsTabThr32);
  M.qs_fast = reinterpret_cast<const QsFast *>(M.qs_tabs + kQsTabFast);
  M.er_bias = e->d_er_bias.as<uint16_t>();
  M.pass_num = (uint32_t)e->model.pass_num;
  M.uniform_bias = e->img.uniform_bias ? 1u : 0u;
  M.method = (uint32_t)e->model.method;
  return M;
}

DeviceGenome device_genome(const pbsim_engine *e) {
  DeviceGenome G;
  G.ascii = e->d_ascii.as<uint8_t>();
  G.pk = e->d_pk.as<uint32_t>();
  G.hp4 = e->d_hp4.as<uint8_t>();
  G.xm = e->d_xm.as<uint32_t>();
  G.len = (uint32_t)e->glen;
  G.seq_num = (uint32_t)e->seq_num;
  return G;
}

DeviceSet device_set(const pbsim_engine *e) {
  DeviceSet S;
  std::memset(&S, 0, sizeof S);
  S.strategy = (uint32_t)e->strategy;
  if (e->strategy == PBSIM_STRATEGY_WGS) return S;
  S.n = (uint32_t)e->set_n;
  S.start = e->d_set_start.as<uint32_t>();
  S.rprefix = e->d_set_rprefix.as<uint64_t>();
  S.plus = e->d_set_plus.as<uint32_t>();
  S.ssp_ends = e->d_set_ssp_ends.as<uint16_t>();
  S.ssp_mod = e->d_set_ssp_mod.as<uint16_t>();
  S.ids = e->d_set_ids.as<uint8_t>();
  S.id_start = e->d_set_idstart.as<uint32_t>();
  S.map_tr = e->replay_map ? e->d_map_tr.as<uint32_t>() : nullptr;
  S.map_k = e->replay_map ? e->d_map_k.as<uint32_t>() : nullptr;
  return S;
}

// bias-dependent threshold tables (re-uploaded with every sequence)
int upload_bias_tables(pbsim_engine *e) {
  e->img.apply_bias(e->model, e->bias);
  if (e->model.method != PBSIM_METHOD_ERRHMM) {
    // thr | qc_prob | thr32 | fast as one block (one bulk copy into shared memory per CTA)
    e->h_qs_tabs.assign(kQsTabBytes, 0);
    std::memcpy(e->h_qs_tabs.data() + kQsTabThr, e->img.qs_thr.data(), PBSIM_NQV * 16);
    std::memcpy(e->h_qs_tabs.data() + kQsTabProb, e->model.qc_prob, PBSIM_NQV * 8);
    std::memcpy(e->h_qs_tabs.data() + kQsTabThr32, e->img.qs_thr32.data(), PBSIM_NQV * 16);
    std::memcpy(e->h_qs_tabs.data() + kQsTabFast, e->img.qs_fast.data(), PBSIM_NQV * 16);
    if (upload(e, e->d_qs_tabs, e->h_qs_tabs.data(), e->h_qs_tabs.size())) return PBSIM_E_CUDA;
    if (upload(e, e->d_qs_thr_hp, e->img.qs_thr_hp.data(), e->img.qs_thr_hp.size())) return PBSIM_E_CUDA;
    if (upload(e, e->d_qs_thr_hp32, e->img.qs_thr_hp32.data(), e->img.qs_thr_hp32.size())) return PBSIM_E_CUDA;
  } else {
    if (upload(e, e->d_er_bias, e->img.er_bias.data(), e->img.er_bias.size())) return PBSIM_E_CUDA;
  }
  CK(cudaStreamSynchronize(e->st));
  return 0;
}

// the sequence text into d_ascii, zero-padded to a multiple of 16 and 64 bytes more; bases == nullptr: a kernel writes it
int upload_ascii(pbsim_engine *e, const char *bases, int64_t len) {
  const size_t padded = ((size_t)len + 15) / 16 * 16 + 64;
  CK(e->d_ascii.ensure(padded));
  CK(cudaMemsetAsync(e->d_ascii.as<uint8_t>() + (len / 16) * 16, 0, padded - (len / 16) * 16, e->st));
  if (bases) CK(cudaMemcpyAsync(e->d_ascii.p, bases, (size_t)len, cudaMemcpyHostToDevice, e->st));
  return 0;
}

// keep_first: sequence sets whose first base keeps its case (see k_set_restore_first)
int finish_sequence_ingest(pbsim_engine *e, int64_t len, int32_t seq_num, const double bias[12], bool keep_first = false) {
  // ascii already in d_ascii (padded with zeros to a multiple of 16)
  const bool set = e->strategy != PBSIM_STRATEGY_WGS;
  e->glen = len;
  e->seq_num = seq_num;
  std::memcpy(e->bias, bias, sizeof e->bias);
  const int64_t words = (len + 15) / 16;
  const int64_t xm_words = ((len >> kXmShift) >> 5) + 2;
  CK(e->d_pk.ensure((size_t)(words + 8) * 4));
  CK(e->d_hp4.ensure((size_t)(len / 2 + 16)));
  CK(e->d_xm.ensure((size_t)xm_words * 4));
  CK(e->d_hpfreq.ensure(12 * 8));
  CK(e->d_biasone.ensure(16));
  CK(e->d_flag.ensure(16));
  CK(cudaMemsetAsync(e->d_xm.p, 0, (size_t)xm_words * 4, e->st));
  CK(cudaMemsetAsync(e->d_hpfreq.p, 0, 12 * 8, e->st));
  CK(cudaMemsetAsync(e->d_flag.p, 0, 16, e->st));
  CK(cudaMemsetAsync(e->d_hp4.p, 0, (size_t)(len / 2 + 16), e->st));
  uint8_t one[16] = {0};
  for (int h = 0; h < 12; ++h) one[h] = (bias[h] == 1.0) ? 1 : 0;
  one[0] = 1;  // hp 0 never occurs inside a sequence
  CK(cudaMemcpyAsync(e->d_biasone.p, one, 16, cudaMemcpyHostToDevice, e->st));
  const uint32_t sn = (uint32_t)e->set_n;
  if (set && keep_first) {
    CK(e->d_set_first.ensure((size_t)sn + 16));
    k_set_save_first<<<nblk(sn, 256), 256, 0, e->st>>>(e->d_ascii.as<uint8_t>(), e->d_set_start.as<uint32_t>(), sn,
                                                       e->d_set_first.as<uint8_t>());
    e->launches++;
  }
  k_upper_pack<<<nblk(words, 256), 256, 0, e->st>>>(e->d_ascii.as<uint8_t>(), len, e->d_pk.as<uint32_t>(),
                                                    e->d_xm.as<uint32_t>());
  if (set) {
    if (keep_first) {
      k_set_restore_first<<<nblk(sn, 256), 256, 0, e->st>>>(e->d_ascii.as<uint8_t>(), e->d_set_start.as<uint32_t>(), sn,
                                                            e->d_set_first.as<uint8_t>(), e->d_pk.as<uint32_t>(),
                                                            e->d_xm.as<uint32_t>());
      e->launches++;
    }
    // transcripts count every base once per read of the transcript (the rprefix differences)
    k_hp_set<<<nblk((len + 1) / 2, 256), 256, 0, e->st>>>(
        e->d_ascii.as<uint8_t>(), len, e->d_set_start.as<uint32_t>(), sn,
        e->strategy == PBSIM_STRATEGY_TRANS ? e->d_set_plus.as<uint32_t>() + sn : nullptr, e->d_hp4.as<uint8_t>(),
        e->d_xm.as<uint32_t>(), e->d_hpfreq.as<unsigned long long>(), e->d_biasone.as<uint8_t>(),
        e->d_flag.as<uint32_t>());
  } else {
    k_hp<<<(unsigned)std::min<int64_t>(nblk((len + 7) / 8, kHpThreads), 148 * 8), kHpThreads, 0, e->st>>>(e->d_ascii.as<uint8_t>(), len, e->d_hp4.as<uint8_t>(),
                                                      e->d_xm.as<uint32_t>(), e->d_hpfreq.as<unsigned long long>(),
                                                      e->d_biasone.as<uint8_t>(), e->d_flag.as<uint32_t>());
  }
  e->launches += 2;
  CK(cudaGetLastError());
  uint32_t flag = 0;
  CK(cudaMemcpyAsync(&flag, e->d_flag.p, 4, cudaMemcpyDeviceToHost, e->st));
  CK(cudaMemcpyAsync(e->hpfreq, e->d_hpfreq.p, 12 * 8, cudaMemcpyDeviceToHost, e->st));
  CK(cudaStreamSynchronize(e->st));
  if (flag) return fail(e, PBSIM_E_INVALID, "sequence holds a homopolymer longer than 65536 bases (unsupported)");
  e->seq_set = true;
  if (e->model_set) return upload_bias_tables(e);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// one batch: plan -> sort -> pass 1 -> quota -> sizes -> emit -> stats
// ---------------------------------------------------------------------------------------------
struct BatchResult {
  uint32_t n_valid_reads = 0;
  bool cut = false;           // a read crossed the quota: the batch ended at n_valid_reads
  uint64_t bases_pass0 = 0;
  uint64_t reads_bytes = 0, maf_bytes = 0;
  uint64_t bases_all = 0;
};

// slices of b_sub_u64, each n_sub + 1 long; kSliceScanIn is the input of a scan (widened counts, pass-0 lengths)
enum U64Slice { kSliceEvOff, kSliceCkOff, kSliceScanIn, kSliceRlen0Prefix, kSliceReadsSize, kSliceMafSize, kSliceNtiles,
                kSliceReadsOff, kSliceMafOff, kSliceTileStart, kSliceSegOff, kSliceChunkOff, kSliceSamSize, kSliceSamOff,
                kU64Slices };

inline unsigned long long *u64_slice(pbsim_engine *e, U64Slice k) {
  return e->b_sub_u64.as<unsigned long long>() + (size_t)k * (e->B.n_sub + 1);
}

int carve_batch(pbsim_engine *e, uint32_t n_reads) {
  const uint32_t pass = (uint32_t)e->model.pass_num;
  const uint64_t n_sub = (uint64_t)n_reads * pass;
  if (n_sub > 0x7FFFFFFFull) return fail(e, PBSIM_E_INVALID, "batch too large");
  CK(e->b_read_u32.ensure((size_t)n_reads * 7 * 4 + 64));
  CK(e->b_sub_u32.ensure((size_t)n_sub * 16 * 4 + 64));
  CK(e->b_sub_u64.ensure((size_t)(n_sub + 1) * kU64Slices * 8 + 64));
  CK(e->b_sub_f64.ensure((size_t)n_sub * 8 + 64));
  Batch &B = e->B;
  B.n_reads = n_reads;
  B.n_sub = (uint32_t)n_sub;
  uint32_t *r32 = e->b_read_u32.as<uint32_t>();
  B.plan_off = r32;
  B.plan_wlen = r32 + n_reads;
  B.plan_raw = r32 + 2ull * n_reads;
  B.plan_meta = r32 + 3ull * n_reads;
  B.plan_tr = r32 + 4ull * n_reads;
  B.grp_copy = r32 + 5ull * n_reads;
  B.grp_num = r32 + 6ull * n_reads;
  uint32_t *s32 = e->b_sub_u32.as<uint32_t>();
  uint32_t **fields[] = {&B.key_in, &B.key_out, &B.idx_in, &B.order, &B.cap, &B.ck_cap, &B.nent, &B.rlen,
                         &B.ncol, &B.nsub, &B.nins, &B.ndel, &B.flags, &B.draws_used, &B.nseg, &B.nchunk};
  for (size_t i = 0; i < sizeof(fields) / sizeof(fields[0]); ++i) *fields[i] = s32 + i * n_sub;
  B.ev_off = reinterpret_cast<uint64_t *>(u64_slice(e, kSliceEvOff));
  B.ck_off = reinterpret_cast<uint64_t *>(u64_slice(e, kSliceCkOff));
  B.accuracy = e->b_sub_f64.as<double>();
  return 0;
}

int excl_scan(pbsim_engine *e, const unsigned long long *in, unsigned long long *out, uint32_t n) {
  size_t tmp = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, (int)n, e->st));
  CK(e->d_cub_tmp.ensure(tmp + 256));
  tmp = e->d_cub_tmp.cap;
  CK(cub::DeviceScan::ExclusiveSum(e->d_cub_tmp.p, tmp, in, out, (int)n, e->st));
  return 0;
}

// out[0..n] = exclusive sum of the uint32 in[0..n), out[n] the total.  tmp holds n + 1 words; the scan reads tmp[n],
// which k_widen does not write and which does not change the sum
int widen_scan(pbsim_engine *e, const uint32_t *in, uint32_t n, unsigned long long *tmp, unsigned long long *out) {
  k_widen<<<nblk(n, 256), 256, 0, e->st>>>(in, n, tmp);
  e->launches++;
  return excl_scan(e, tmp, out, n + 1);
}

int sort_pairs(pbsim_engine *e, const uint32_t *keys_in, uint32_t *keys_out, const uint32_t *vals_in, uint32_t *vals_out,
               uint32_t n, int begin_bit, int end_bit) {
  size_t tmp = 0;
  CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys_in, keys_out, vals_in, vals_out, (int)n, begin_bit, end_bit, e->st));
  CK(e->d_cub_tmp.ensure(tmp + 256));
  tmp = e->d_cub_tmp.cap;
  CK(cub::DeviceRadixSort::SortPairs(e->d_cub_tmp.p, tmp, keys_in, keys_out, vals_in, vals_out, (int)n, begin_bit, end_bit,
                                     e->st));
  return 0;
}

// the CTAs of one pass: bin b (accuracy * 2 + slow, sim_kernels.cuh) holds the sorted items
// [bin_lo[b], bin_hi[b]) and owns the CTAs from cta_first[b]; CTA slot i runs CTA order[i]
struct CtaSchedule {
  uint32_t *bin_start, *bin_lo, *bin_hi, *cta_first, *order;
  uint32_t slots;
};

// Sorts the items by key bits [begin_bit, 28) (ids_out: the items in that order), bins them and maps the bins to CTAs
// of cta_threads items.  longest_first orders the CTAs by their first key (k_cta_keys), otherwise they run in bin
// order.  The arrays are carved from buf.  Counts its 4 launches; CUB's are not counted.
int schedule_ctas(pbsim_engine *e, DevBuf &buf, const uint32_t *keys_in, uint32_t *keys_out, const uint32_t *ids_in,
                  uint32_t *ids_out, uint32_t n, int begin_bit, uint32_t cta_threads, bool longest_first,
                  CtaSchedule *s) {
  s->slots = nblk(n, cta_threads) + kBins;
  CK(buf.ensure((4 * kBins + 8) * 4 + (size_t)s->slots * 4 * 4 + 64));
  s->bin_start = buf.as<uint32_t>();
  s->bin_lo = s->bin_start + kBins + 1;
  s->bin_hi = s->bin_lo + kBins;
  s->cta_first = s->bin_hi + kBins;
  uint32_t *cta_key = s->cta_first + kBins + 1, *cta_id = cta_key + s->slots, *cta_key_s = cta_id + s->slots;
  s->order = cta_key_s + s->slots;
  int rc = sort_pairs(e, keys_in, keys_out, ids_in, ids_out, n, begin_bit, 28);
  if (rc) return rc;
  k_fill_u32<<<1, 256, 0, e->st>>>(s->bin_start, kBins + 1, 0xFFFFFFFFu);
  k_bin_bounds<<<nblk(n, 256), 256, 0, e->st>>>(keys_out, n, s->bin_start);
  k_cta_map<<<1, 32, 0, e->st>>>(s->bin_start, keys_out, n, s->bin_lo, s->bin_hi, s->cta_first, cta_threads);
  e->launches += 4;
  if (!longest_first) {
    k_iota_u32<<<nblk(s->slots, 256), 256, 0, e->st>>>(s->order, s->slots);
    return 0;
  }
  k_cta_keys<<<nblk(s->slots, 256), 256, 0, e->st>>>(keys_out, s->bin_lo, s->cta_first, s->slots, cta_key, cta_id,
                                                    cta_threads);
  return sort_pairs(e, cta_key, cta_key_s, cta_id, s->order, s->slots, 0, 21);
}

// the CTA map of a schedule in kernel arguments (SimArgs, SegArgs)
template <class Args>
void set_ctas(Args &a, const CtaSchedule &s) {
  a.cta_order = s.order;
  a.cta_first = s.cta_first;
  a.bin_lo = s.bin_lo;
  a.bin_hi = s.bin_hi;
}

// what the phases of one batch share besides the engine and its batch arrays (e->B)
struct BatchCtx {
  uint32_t pass, cta_threads;
  int64_t clip_room;       // >= 0: the one read of a tail batch is clipped to this many bases
  const SampleBatch *sb;   // --method sample: the groups of this batch (n_reads = their copies); otherwise null
  bool qs, sample, spec, replay;
  DevicePool Pl;
  SimArgs A;                 // pass-1 arguments; their model M, genome G and generator rng serve every phase
  int64_t next_start_after = -1;  // replay: draw-log start of the subread behind the batch (-1: none)
  // the current attempt
  bool use_segments;
  CtaSchedule cta;  // pass-1 CTAs of the sub-reads
  uint64_t n_seg_total, n_chunk_total;
};

inline unsigned long long *host_ctrl(pbsim_engine *e) { return reinterpret_cast<unsigned long long *>(e->h_ctrl.p); }

// replay: upload the slice of the draw log this batch can touch
int upload_replay_window(pbsim_engine *e, BatchCtx &c) {
  const int64_t s0 = (int64_t)(e->next_read - e->run.first_read) * c.pass, n_sub = e->B.n_sub;
  if (s0 + n_sub > e->run.replay_nsubreads)
    return fail(e, PBSIM_E_REPLAY, "replay log exhausted: batch needs subreads %lld..%lld but the log has %lld",
                (long long)s0, (long long)(s0 + n_sub), (long long)e->run.replay_nsubreads);
  const int64_t d0 = e->run.replay_starts[s0];
  const int64_t d1 = (s0 + n_sub < e->run.replay_nsubreads) ? e->run.replay_starts[s0 + n_sub] : e->run.replay_ndraws;
  c.next_start_after = (s0 + n_sub < e->run.replay_nsubreads) ? d1 : e->run.replay_ndraws;
  if (d0 < 0 || d1 < d0 || d1 > e->run.replay_ndraws) return fail(e, PBSIM_E_REPLAY, "replay starts are not monotone");
  if (upload(e, e->d_draws, e->run.replay_draws + d0, (size_t)(d1 - d0))) return PBSIM_E_CUDA;
  if (upload(e, e->d_starts, e->run.replay_starts + s0, (size_t)n_sub)) return PBSIM_E_CUDA;
  c.A.rng.draws = e->d_draws.as<int32_t>();
  c.A.rng.draws_base = d0;
  c.A.rng.draws_end = d1;
  c.A.rng.starts = e->d_starts.as<int64_t>();
  return 0;
}

// K1 plan, then the pass-1 schedule: sub-reads sorted by (accuracy, length desc), longest-first CTA order
int plan(pbsim_engine *e, BatchCtx &c) {
  Batch &B = e->B;
  const uint32_t seg_min_len = c.use_segments ? (uint32_t)e->seg_min_len : 0u;
  if (c.sample)
    k_plan_sample<<<nblk(B.n_reads, 256), 256, 0, e->st>>>(c.A.G, c.Pl, *c.sb, B, e->cap_num, e->cap_den, c.spec ? 1u : 0u,
                                                             c.A.rng.seed, c.A.M.uniform_bias ? 1u : 0u, seg_min_len);
  else
    k_plan<<<nblk(B.n_reads, 256), 256, 0, e->st>>>(c.A.M, c.A.G, device_set(e), c.A.rng, B, c.clip_room, e->cap_num,
                                                      e->cap_den, c.qs ? 8u : 16u, seg_min_len, e->seg_extra,
                                                      e->chain_chunk_eff());
  e->launches++;
  return schedule_ctas(e, e->d_bins, B.key_in, B.key_out, B.idx_in, B.order, B.n_sub, 0, c.cta_threads, true, &c.cta);
}

// event and checkpoint slots, and with segments the segment and chunk lists: offsets by scans, totals read back
int size_slots(pbsim_engine *e, BatchCtx &c) {
  Batch &B = e->B;
  unsigned long long *hctrl = host_ctrl(e);
  unsigned long long *tmp = u64_slice(e, kSliceScanIn);
  unsigned long long *seg_off = u64_slice(e, kSliceSegOff), *chunk_off = u64_slice(e, kSliceChunkOff);
  int rc;
  if ((rc = widen_scan(e, B.cap, B.n_sub, tmp, reinterpret_cast<unsigned long long *>(B.ev_off)))) return rc;
  if ((rc = widen_scan(e, B.ck_cap, B.n_sub, tmp, reinterpret_cast<unsigned long long *>(B.ck_off)))) return rc;
  if (c.use_segments) {
    if ((rc = widen_scan(e, B.nseg, B.n_sub, tmp, seg_off))) return rc;
    if (peek(e, hctrl + 2, seg_off + B.n_sub, 8)) return PBSIM_E_CUDA;
    if ((rc = widen_scan(e, B.nchunk, B.n_sub, tmp, chunk_off))) return rc;
    if (peek(e, hctrl + 4, chunk_off + B.n_sub, 8)) return PBSIM_E_CUDA;
  }
  if (peek(e, hctrl, B.ev_off + B.n_sub, 8)) return PBSIM_E_CUDA;
  if (peek(e, hctrl + 1, B.ck_off + B.n_sub, 8)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  c.n_seg_total = c.use_segments ? hctrl[2] : 0;
  c.n_chunk_total = c.use_segments ? hctrl[4] : 0;
  if (c.n_seg_total > 0x7FFFFFF0ull) return fail(e, PBSIM_E_INVALID, "too many segments in one batch");
  CK(e->d_ev.ensure((size_t)hctrl[0] * (c.qs ? 2 : 1) + 256));
  CK(e->d_ck.ensure((size_t)hctrl[1] * sizeof(Ckpt) + 256));
  if (c.n_seg_total > 0) CK(e->d_seg.ensure((size_t)c.n_seg_total * (6 * 4 + sizeof(SegResult)) + 256));
  return 0;
}

// K2 / K3: sequential pass 1, one thread per sub-read
void pass1_sequential(pbsim_engine *e, BatchCtx &c) {
  SimArgs &A = c.A;
  set_ctas(A, c.cta);
  A.ev = e->d_ev.as<uint8_t>();
  A.ck = e->d_ck.as<Ckpt>();
  const uint32_t grid = c.cta.slots;
  if (c.sample) {
    if (c.replay) k_sim_sample<PBSIM_RNG_REPLAY><<<grid, kSimThreads, 0, e->st>>>(A, c.Pl, *c.sb, 0u);
    else k_sim_sample<PBSIM_RNG_PHILOX><<<grid, kSimThreads, 0, e->st>>>(A, c.Pl, *c.sb, 0u);
  } else if (c.qs) {
    if (c.replay) k_sim_qshmm<PBSIM_RNG_REPLAY><<<grid, kSimThreads, kQsSmemBytes, e->st>>>(A);
    else k_sim_qshmm<PBSIM_RNG_PHILOX><<<grid, kSimThreads, kQsSmemBytes, e->st>>>(A);
  } else {
    const uint32_t smem = e->er_smem_bar_off + 16;
    if (c.replay) k_sim_errhmm<PBSIM_RNG_REPLAY><<<grid, kErrThreads, smem, e->st>>>(A, e->er_smem_bar_off);
    else k_sim_errhmm<PBSIM_RNG_PHILOX><<<grid, kErrThreads, smem, e->st>>>(A, e->er_smem_bar_off);
  }
  e->launches++;
}

// segment-parallel pass 1 for the long reads (seg_kernels.cuh): chain chunks recover the HMM state in front of their
// segments (qshmm model accuracies: and simulate them, k_qs_pass1), the other segments run (k_sim_seg, k_sim_seg_err)
// and k_find_end finds where each read ends
int pass1_segments(pbsim_engine *e, BatchCtx &c) {
  const Batch &B = e->B;
  const uint32_t nseg = (uint32_t)c.n_seg_total;
  SegBatch S;
  S.n_seg_total = nseg;
  S.seg_off = reinterpret_cast<const uint64_t *>(u64_slice(e, kSliceSegOff));
  S.seg_res = e->d_seg.as<SegResult>();
  uint32_t *u = reinterpret_cast<uint32_t *>(S.seg_res + nseg);
  uint32_t **seg_arrays[] = {&S.seg_sub, &S.seg_key_in, &S.seg_key_out, &S.seg_id_in, &S.seg_order, &S.seg_state};
  for (size_t i = 0; i < 6; ++i) *seg_arrays[i] = u + i * nseg;
  // qshmm: k_qs_pass1 simulates the segments of model accuracies, k_sim_seg the others (if the model has accuracies
  // without a chain) and those of --method sample
  bool freq_only = false;
  for (const AccEntry &a : e->img.acc) freq_only |= a.valid && !a.has_model;
  const bool seg_pass = !c.qs || c.sample || freq_only;
  k_seg_fill<<<nblk(B.n_sub, 256), 256, 0, e->st>>>(B, S, c.pass, c.qs && !c.sample ? 1u : 0u);
  CtaSchedule sc = {};
  int rc = 0;
  if (seg_pass && (rc = schedule_ctas(e, e->d_seg_bins, S.seg_key_in, S.seg_key_out, S.seg_id_in, S.seg_order, nseg, 20,
                                      c.cta_threads, false, &sc)))
    return rc;
  SegArgs SA;
  SA.keys = c.A.keys;
  SA.M = c.A.M;
  SA.G = c.A.G;
  SA.bias_one = e->d_biasone.as<uint8_t>();
  SA.B = B;
  SA.S = S;
  set_ctas(SA, sc);
  SA.ev = e->d_ev.as<uint8_t>();
  SA.pool_q = c.Pl.quals;
  SA.pool_start = c.Pl.start;
  if (c.n_chunk_total > 0) {
    const uint32_t nch = (uint32_t)c.n_chunk_total;
    const uint32_t chain_threads = c.qs ? (uint32_t)kChainThreads : c.cta_threads;
    CK(e->d_chunk.ensure((size_t)nch * 5 * 4 + 64));
    ChunkBatch C;
    C.n_chunks = nch;
    C.per_chunk = e->chain_chunk_eff();
    C.qs = c.qs ? 1u : 0u;
    C.chunk_off = reinterpret_cast<const uint64_t *>(u64_slice(e, kSliceChunkOff));
    uint32_t **chunk_arrays[] = {&C.sub, &C.key_in, &C.key_out, &C.id_in, &C.order};
    for (size_t i = 0; i < 5; ++i) *chunk_arrays[i] = e->d_chunk.as<uint32_t>() + i * nch;
    k_chunk_fill<<<nblk(B.n_sub, 256), 256, 0, e->st>>>(B, C, c.pass);
    CtaSchedule cc;
    if ((rc = schedule_ctas(e, e->d_chunk_bins, C.key_in, C.key_out, C.id_in, C.order, nch, 0, chain_threads, true, &cc)))
      return rc;
    SegArgs CA = SA;
    set_ctas(CA, cc);
    CK(cudaEventRecord(e->ev_chain[0], e->st));
    if (c.qs) k_qs_pass1<<<cc.slots, kChainThreads, kQsSmemBytes, e->st>>>(CA, C);
    else k_chain_chunk_err<<<cc.slots, kErrThreads, e->er_smem_bar_off + 16, e->st>>>(CA, C, e->er_smem_bar_off);
    CK(cudaEventRecord(e->ev_chain[1], e->st));
    e->launches += 2;
  }
  CK(cudaEventRecord(e->ev_seg[0], e->st));
  const uint32_t end_grid = nblk((uint64_t)B.n_sub * 32, 128);
  if (c.qs) {
    if (c.sample) k_sim_seg<true><<<sc.slots, kSimThreads, 0, e->st>>>(SA);
    else if (seg_pass) k_sim_seg<false><<<sc.slots, kSimThreads, 0, e->st>>>(SA);
    e->launches += seg_pass ? 1 : 0;
    CK(cudaEventRecord(e->ev_seg[1], e->st));
    k_find_end<<<end_grid, 128, 0, e->st>>>(B, S, c.A.G, SA.bias_one, c.pass, SA.ev, e->d_ck.as<Ckpt>(), c.A.M.qs_fast,
                                            c.sample ? 1u : 0u);
  } else {
    k_sim_seg_err<<<sc.slots, kErrThreads, e->er_smem_bar_off + 16, e->st>>>(SA, e->er_smem_bar_off);
    CK(cudaEventRecord(e->ev_seg[1], e->st));
    k_find_end_err<<<end_grid, 128, 0, e->st>>>(B, S, c.A.G, SA.keys, SA.bias_one, c.pass, SA.ev, e->d_ck.as<Ckpt>());
    e->launches++;
  }
  e->launches += 2;
  e->seg_batches++;
  return 0;
}

// --method sample: which copies assumed a wrong length?  Their groups' tails are redone as chains (k_sample_redo), one
// thread per chain, in the sequential slot layout (k_sim_sample clears the reads' "segmented" mark)
int sample_redo(pbsim_engine *e, BatchCtx &c) {
  Batch &B = e->B;
  unsigned long long *ctrl = e->d_ctrl.as<unsigned long long>(), *hctrl = host_ctrl(e);
  hctrl[6] = 0;
  CK(cudaMemsetAsync(ctrl + 6, 0, 8, e->st));
  k_sample_redo<<<nblk(B.n_reads, 256), 256, 0, e->st>>>(B, ctrl + 6);
  if (peek(e, hctrl + 6, ctrl + 6, 8)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  e->launches += 2;
  if (hctrl[6] == 0) return 0;
  const int rc =
      schedule_ctas(e, e->d_bins, B.key_in, B.key_out, B.idx_in, B.order, B.n_sub, 0, c.cta_threads, true, &c.cta);
  if (rc) return rc;
  if (c.replay) k_sim_sample<PBSIM_RNG_REPLAY><<<c.cta.slots, kSimThreads, 0, e->st>>>(c.A, c.Pl, *c.sb, 1u);
  else k_sim_sample<PBSIM_RNG_PHILOX><<<c.cta.slots, kSimThreads, 0, e->st>>>(c.A, c.Pl, *c.sb, 1u);
  e->launches++;
  e->sample_redo_groups += (int64_t)hctrl[6];
  if (hctrl[6] * 2 > c.sb->n_groups) e->sample_spec_run = false;  // deletion-rich mix: chains from the start
  return 0;
}

// which read crosses len_quota: waits for pass 1 and reads back hctrl[0] the cut, [1] the pass-0 bases in front of
// it, [2] the pass-1 flags, [3] replay: the subreads whose draws disagree with the log
int quota_cut(pbsim_engine *e, BatchCtx &c, int attempt) {
  const Batch &B = e->B;
  const uint32_t n_reads = B.n_reads, n_sub = B.n_sub;
  unsigned long long *ctrl = e->d_ctrl.as<unsigned long long>(), *hctrl = host_ctrl(e);
  unsigned long long *rl0 = u64_slice(e, kSliceScanIn);
  unsigned long long *prefix = u64_slice(e, kSliceRlen0Prefix);
  k_rlen0<<<nblk(n_reads, 256), 256, 0, e->st>>>(B.rlen, n_reads, c.pass, rl0);
  const int rc = excl_scan(e, rl0, prefix, n_reads);
  if (rc) return rc;
  hctrl[0] = n_reads;
  hctrl[1] = 0;
  hctrl[2] = 0;
  hctrl[3] = 0;
  CK(cudaMemcpyAsync(ctrl, hctrl, 32, cudaMemcpyHostToDevice, e->st));
  if (c.sample)
    k_find_cut_sample<<<nblk(n_reads, 256), 256, 0, e->st>>>(prefix, n_reads, e->len_total, e->run.len_quota, ctrl);
  else if (c.clip_room < 0)  // bulk batch: speculative unclipped plans
    k_find_cut<<<nblk(n_reads, 256), 256, 0, e->st>>>(prefix, B.plan_raw, n_reads, e->len_total, e->run.len_quota, ctrl);
  k_batch_totals<<<nblk(n_sub, 256), 256, 0, e->st>>>(prefix, B.rlen, B.flags, n_reads, c.pass, ctrl);
  e->launches += 3;
  if (c.replay) {
    k_check_replay<<<nblk(n_sub, 256), 256, 0, e->st>>>(c.A.rng.starts, B.draws_used, B.plan_wlen, (uint32_t)e->glen, n_sub,
                                                        c.pass, c.next_start_after, ctrl,
                                                        reinterpret_cast<unsigned int *>(&ctrl[3]));
    e->launches++;
  }
  if (peek(e, hctrl, ctrl, 32)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  const uint32_t flags = (uint32_t)hctrl[2];
  if (flags & 2u) return fail(e, PBSIM_E_PARAM, "a read drew an accuracy for which the model has no usable tables");
  float pass1_ms = 0, ms = 0;
  CK(cudaEventElapsedTime(&pass1_ms, e->ev_k[0], e->ev_k[1]));
  e->sim_ms += pass1_ms;
  if (c.n_seg_total > 0) {
    CK(cudaEventElapsedTime(&ms, e->ev_seg[0], e->ev_seg[1]));
    e->seg_ms += ms;
    if (c.n_chunk_total > 0) {
      CK(cudaEventElapsedTime(&ms, e->ev_chain[0], e->ev_chain[1]));
      e->chain_ms += ms;
    }
  }
  if (getenv("PBSIM_DEBUG"))
    fprintf(stderr, "[pbsim] batch reads=%u sub=%u segments=%llu flags=%u pass1_ms=%.2f attempt=%d\n", n_reads, n_sub,
            (unsigned long long)c.n_seg_total, flags, pass1_ms, attempt);
  return 0;
}

// K5 (option "align"): the MAF blocks pass 2 left in d_aln_maf -> SAM alignment lines in the output set's second stream
int align_batch(pbsim_engine *e, const EmitArgs &EA, BatchResult *out) {
  const uint32_t n = EA.n_sub;
  unsigned long long *sam_size = u64_slice(e, kSliceSamSize), *sam_off = u64_slice(e, kSliceSamOff);
  CK(cudaMemsetAsync(sam_size + n, 0, 8, e->st));
  CK(e->d_aln_rec.ensure((size_t)n * sizeof(AlnRec) + 64));
  AlnArgs A;
  A.S = EA.S;
  A.B = EA.B;
  A.P = EA.P;
  A.n_sub = n;
  A.lay = EA.lay;
  A.reads_off = EA.reads_off;
  A.maf_off = EA.maf_off;
  A.reads = EA.out_reads;
  A.maf = EA.out_maf;
  A.rname = e->d_rname.as<uint8_t>();
  A.rname_len = (uint32_t)e->seq_name.size();
  A.rec = e->d_aln_rec.as<AlnRec>();
  A.sam_off = (const uint64_t *)sam_off;
  A.sam = nullptr;
  const uint32_t grid = nblk(n, 8);
  k_aln_sizes<<<grid, 256, 0, e->st>>>(A, (uint64_t *)sam_size);
  e->launches++;
  int rc;
  if ((rc = excl_scan(e, sam_size, sam_off, n + 1))) return rc;
  unsigned long long *hctrl = host_ctrl(e);
  if (peek(e, hctrl + 11, sam_off + n, 8)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  out->maf_bytes = hctrl[11];
  pbsim_engine::OutSet &O = e->out[e->cur_set];
  CK(O.maf.ensure((size_t)out->maf_bytes + 256));
  A.sam = O.maf.as<uint8_t>();
  k_aln_write<<<grid, 256, 0, e->st>>>(A);
  e->launches++;
  return 0;
}

// K4 record sizes, offsets and text of the reads before the cut, K6 their statistics, and the read-back of their
// accuracies and lengths
int emit_batch(pbsim_engine *e, const BatchCtx &c, BatchResult *out) {
  const Batch &B = e->B;
  const uint32_t nv_sub = out->n_valid_reads * c.pass;
  if (nv_sub == 0) return 0;
  unsigned long long *hctrl = host_ctrl(e);

  // ---- K4 sizes + offsets
  unsigned long long *reads_size = u64_slice(e, kSliceReadsSize);
  unsigned long long *maf_size = u64_slice(e, kSliceMafSize);
  unsigned long long *ntiles = u64_slice(e, kSliceNtiles);
  unsigned long long *reads_off = u64_slice(e, kSliceReadsOff);
  unsigned long long *maf_off = u64_slice(e, kSliceMafOff);
  unsigned long long *tile_start = u64_slice(e, kSliceTileStart);
  CK(cudaMemsetAsync(reads_size + nv_sub, 0, 8, e->st));
  CK(cudaMemsetAsync(maf_size + nv_sub, 0, 8, e->st));
  CK(cudaMemsetAsync(ntiles + nv_sub, 0, 8, e->st));
  e->emitp.glen = (uint32_t)e->glen;
  e->emitp.sam = e->model.pass_num > 1 ? (e->bam ? 2u : 1u) : 0u;
  e->emitp.qs_segments = c.qs ? 1u : 0u;
  e->emitp.sample = c.sample ? 1u : 0u;
  {
    char head[192];
    if (e->strategy == PBSIM_STRATEGY_WGS) snprintf(head, sizeof head, "%s%d", e->model.id_prefix, e->seq_num);
    else snprintf(head, sizeof head, "%s", e->model.id_prefix);  // "<prefix>_<read>" (:2951, :3469)
    e->emitp.id_head_len = (uint32_t)strlen(head);
    memcpy(e->emitp.id_head, head, e->emitp.id_head_len + 1);
  }
  CK(e->d_lay.ensure((size_t)nv_sub * sizeof(EmitLay) + 64));
  k_sizes<<<nblk(nv_sub, 256), 256, 0, e->st>>>(B, e->emitp, device_set(e), nv_sub, (uint64_t *)reads_size, (uint64_t *)maf_size,
                                                (uint64_t *)ntiles, e->d_lay.as<EmitLay>());
  e->launches++;
  int rc;
  if ((rc = excl_scan(e, reads_size, reads_off, nv_sub + 1))) return rc;
  if ((rc = excl_scan(e, maf_size, maf_off, nv_sub + 1))) return rc;
  if ((rc = excl_scan(e, ntiles, tile_start, nv_sub + 1))) return rc;
  if (peek(e, hctrl + 8, reads_off + nv_sub, 8)) return PBSIM_E_CUDA;
  if (peek(e, hctrl + 9, maf_off + nv_sub, 8)) return PBSIM_E_CUDA;
  if (peek(e, hctrl + 10, tile_start + nv_sub, 8)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  out->reads_bytes = hctrl[8];
  out->maf_bytes = hctrl[9];
  const uint64_t n_tiles = hctrl[10];
  pbsim_engine::OutSet &O = e->out[e->cur_set];
  CK(O.reads.ensure((size_t)out->reads_bytes + 256));
  // option "align": the MAF blocks go to a scratch stream, from which k_aln_* write the alignment lines into O.maf
  DevBuf &maf_buf = e->align ? e->d_aln_maf : O.maf;
  CK(maf_buf.ensure((size_t)out->maf_bytes + 256));

  // ---- K4 emit
  EmitArgs EA;
  EA.S = device_set(e);
  EA.G = c.A.G;
  EA.B = B;
  EA.P = e->emitp;
  EA.ev = e->d_ev.as<uint8_t>();
  EA.ck = e->d_ck.as<Ckpt>();
  EA.n_sub = nv_sub;
  EA.n_tiles = n_tiles;
  EA.tile_start = (const uint64_t *)tile_start;
  CK(e->d_tile_sub.ensure((size_t)n_tiles * 4 + 64));
  CK(e->d_tile_desc.ensure((size_t)n_tiles * sizeof(TileDesc) + 64));
  EA.tile_sub = e->d_tile_sub.as<uint32_t>();
  EA.desc = e->d_tile_desc.as<TileDesc>();
  EA.lay = e->d_lay.as<EmitLay>();
  EA.reads_off = (const uint64_t *)reads_off;
  EA.maf_off = (const uint64_t *)maf_off;
  EA.keys.init(e->run.seed, (uint32_t)e->seq_num);
  EA.philox = c.replay ? 0u : 1u;
  EA.out_reads = O.reads.as<uint8_t>();
  EA.out_maf = maf_buf.as<uint8_t>();
  if (n_tiles > 0) {
    int dev_sms = 148;
    cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, e->device);
    const uint64_t want = (n_tiles + kEmitWarps - 1) / kEmitWarps;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(want, (uint64_t)dev_sms * 8 * 4);
    CK(cudaEventRecord(e->ev_k[2], e->st));
    // per-tile descriptors (and the tile -> sub-read map), then the row kernel on the plain text tiles and
    // k_emit on everything else (headers, exceptional / wide tiles, SAM arrays, BAM records)
    if (c.qs) k_tile_desc<PBSIM_METHOD_QSHMM><<<nblk(n_tiles, 256), 256, 0, e->st>>>(EA, e->d_tile_sub.as<uint32_t>());
    else k_tile_desc<PBSIM_METHOD_ERRHMM><<<nblk(n_tiles, 256), 256, 0, e->st>>>(EA, e->d_tile_sub.as<uint32_t>());
    e->launches++;
    if (EA.P.sam == 2u) {  // BAM packs bases with atomic ORs: the records start zeroed
      CK(cudaMemsetAsync(O.reads.p, 0, (size_t)out->reads_bytes, e->st));
      if (c.qs) k_emit<PBSIM_METHOD_QSHMM, true><<<grid, kEmitThreads, 0, e->st>>>(EA);
      else k_emit<PBSIM_METHOD_ERRHMM, true><<<grid, kEmitThreads, 0, e->st>>>(EA);
    } else {
      const uint32_t glen_words = (uint32_t)((e->glen + 15) / 16);
      if (c.qs) {
        k_emit_rows<PBSIM_METHOD_QSHMM><<<grid, kEmitThreads, 0, e->st>>>(EA.desc, n_tiles, EA.ev, c.A.G.pk, glen_words, EA.out_reads, EA.out_maf);
        k_emit<PBSIM_METHOD_QSHMM, false><<<grid, kEmitThreads, 0, e->st>>>(EA);
      } else {
        k_emit_rows<PBSIM_METHOD_ERRHMM><<<grid, kEmitThreads, 0, e->st>>>(EA.desc, n_tiles, EA.ev, c.A.G.pk, glen_words, EA.out_reads, EA.out_maf);
        k_emit<PBSIM_METHOD_ERRHMM, false><<<grid, kEmitThreads, 0, e->st>>>(EA);
      }
      e->launches++;
    }
    if (e->align && (rc = align_batch(e, EA, out))) return rc;
    CK(cudaEventRecord(e->ev_k[3], e->st));
    e->launches++;
  }
  // ---- K6 stats
  k_stats<<<nblk(nv_sub, 256), 256, 0, e->st>>>(B, nv_sub, c.pass, e->d_stats.as<unsigned long long>(), e->freq_len_cells);
  e->launches++;
  CK(cudaGetLastError());

  // per-subread accuracy values: summed on the host in read order (accuracy_total, :2314)
  CK(e->h_acc.ensure((size_t)nv_sub * 8 + (size_t)nv_sub * 4 * 3 + 64));
  double *hacc = reinterpret_cast<double *>(e->h_acc.p);
  uint32_t *hrlen = reinterpret_cast<uint32_t *>(hacc + nv_sub);
  if (peek(e, hacc, B.accuracy, (size_t)nv_sub * 8)) return PBSIM_E_CUDA;
  if (peek(e, hrlen, B.rlen, (size_t)nv_sub * 4)) return PBSIM_E_CUDA;
  return 0;
}

// sb: --method sample, the groups of this batch (n_reads = their copies); otherwise null
int run_batch(pbsim_engine *e, uint32_t n_reads, int64_t clip_room, BatchResult *out, const SampleBatch *sb = nullptr) {
  BatchCtx c = {};
  c.pass = (uint32_t)e->model.pass_num;
  c.qs = e->model.method != PBSIM_METHOD_ERRHMM;  // sample reads use the qshmm event stream
  c.sample = e->model.method == PBSIM_METHOD_SAMPLE;
  c.cta_threads = c.qs ? kSimThreads : kErrThreads;
  c.Pl = {e->d_pool_q.as<uint8_t>(), e->d_pool_start.as<uint64_t>(),
          (uint32_t)(e->pool_start.empty() ? 0 : e->pool_start.size() - 1)};
  if (c.sample && !sb) return fail(e, PBSIM_E_INVALID, "internal: sample batch without groups");
  c.sb = sb;
  c.spec = c.sample && e->sample_spec && e->sample_spec_run;
  c.replay = e->run.rng_mode == PBSIM_RNG_REPLAY;
  c.clip_room = clip_room;
  int rc = carve_batch(e, n_reads);
  if (rc) return rc;
  e->B.first_read = (uint64_t)e->next_read;
  CK(e->d_ctrl.ensure(64 * 8));
  CK(e->h_ctrl.ensure(64 * 8));
  const unsigned long long *hctrl = host_ctrl(e);
  SimArgs &A = c.A;  // what stays the same over the attempts
  A.bias_one = e->d_biasone.as<uint8_t>();
  A.plan_draws = e->strategy == PBSIM_STRATEGY_TRANS ? 3u : (e->strategy == PBSIM_STRATEGY_TEMPL ? 1u : 0u);
  A.keys.init(e->run.seed, (uint32_t)e->seq_num);
  A.M = device_model(e);
  A.G = device_genome(e);
  A.rng.mode = (uint32_t)e->run.rng_mode;
  A.rng.seed = e->run.seed;  // the draw log of replay: upload_replay_window
  A.B = e->B;
  if (c.replay && (rc = upload_replay_window(e, c))) return rc;

  // (the single, quota-clipped read of a tail batch is segmented too: on one thread a 50 kb read takes milliseconds)
  // (--method sample: the speculative pass of PHILOX runs; the chains that have to be redone stay sequential)
  c.use_segments = !c.replay && e->seg_enabled && (!c.sample || c.spec);
  int seg_retries = 0;
  for (int attempt = 0; attempt < 9; ++attempt) {
    if ((rc = plan(e, c))) return rc;
    if ((rc = size_slots(e, c))) return rc;
    CK(cudaEventRecord(e->ev_k[0], e->st));
    pass1_sequential(e, c);
    if (c.n_seg_total > 0 && (rc = pass1_segments(e, c))) return rc;
    if (c.spec && (rc = sample_redo(e, c))) return rc;
    CK(cudaEventRecord(e->ev_k[1], e->st));
    CK(cudaGetLastError());
    if ((rc = quota_cut(e, c, attempt))) return rc;
    const uint32_t flags = (uint32_t)hctrl[2];
    if (flags & 4u) {
      // A segmented read could not be completed.  If the only reason is that its window outlasted the segments
      // provisioned for it (a read that stays in an insertion-rich state of a sticky chain), provision more — the
      // headroom stays for the batches to come; anything else redoes the batch on the sequential path.
      const uint32_t inner = flags >> 8;
      if (inner == 4u && e->seg_extra < 0.6f && seg_retries < 3) {
        e->seg_extra += 0.04f;
        ++seg_retries;
        continue;
      }
      c.use_segments = false;
      e->seg_fallback_batches++;
      if (attempt >= 8) return fail(e, PBSIM_E_OVERFLOW, "segment-parallel pass 1 failed repeatedly");
      continue;
    }
    if (flags & 1u) {  // a read outgrew its slot: enlarge and redo the batch
      e->cap_num *= 2;
      if (attempt >= 8) return fail(e, PBSIM_E_OVERFLOW, "event slots overflowed repeatedly");
      continue;
    }
    const uint64_t cut = hctrl[0];
    out->cut = cut < n_reads;
    out->n_valid_reads = out->cut ? (uint32_t)cut : n_reads;
    out->bases_pass0 = hctrl[1];
    if (c.replay && hctrl[3] != 0)
      return fail(e, PBSIM_E_REPLAY, "replay: %llu subreads consumed a different number of draws than the log says",
                  (unsigned long long)hctrl[3]);
    break;
  }
  return emit_batch(e, c, out);
}

// ---------------------------------------------------------------------------------------------
// batch production (the quota loop of pbsim.cpp:2173 / :3792 in batches) and delivery
// ---------------------------------------------------------------------------------------------

// k_gz_encode's dynamic shared memory: above the 48 KB a launch gets without asking (set in pbsim_cuda_create)
constexpr size_t kGzEncodeSmem = (size_t)kGzImgWords * 4 + kGzCodes * 256 * 4;

// gzip one record stream of the batch in HBM (gz_kernels.cuh): histogram -> code (host) -> member sizes -> offsets
// -> members.  Replaces the reference's popen("gzip > file") children (pbsim.cpp:708-730).
int gz_compress(pbsim_engine *e, const uint8_t *in, uint64_t n, DevBuf &dst, uint64_t *out_bytes, bool bgzf = false) {
  *out_bytes = 0;
  if (n == 0) return 0;
  static_assert(sizeof(GzTables) % 8 == 0, "GzTables is copied as words");
  CK(e->d_gz_hist.ensure(512 * 8));
  CK(e->d_gz_tables.ensure(sizeof(GzTables)));
  CK(e->h_gz.ensure(512 * 8 + sizeof(GzTables) + 64));
  unsigned long long *hh = reinterpret_cast<unsigned long long *>(e->h_gz.p);
  GzTables *ht = reinterpret_cast<GzTables *>(hh + 512);
  CK(cudaMemsetAsync(e->d_gz_hist.p, 0, 512 * 8, e->st));
  int dev_sms = 148;
  cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, e->device);
  // streams above 64 MiB are sampled: one 16-byte chunk in 16
  k_gz_hist<<<(uint32_t)std::min<uint64_t>((n + 4095) / 4096, (uint64_t)dev_sms * 8), 256, 0, e->st>>>(
      in, n, n > ((uint64_t)64 << 20) ? 16u : 1u, e->d_gz_hist.as<unsigned long long>());
  e->launches++;
  if (peek(e, hh, e->d_gz_hist.p, 512 * 8)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  {
    // three codes per stream: code 0 from the sequence-like text, code 1 from the rest, code 2 from all of it
    // (gz_kernels.cuh)
    std::memset(ht, 0, sizeof *ht);
    for (uint32_t c = 0; c < kGzCodes; ++c) {
      uint64_t hist[256];
      for (int i = 0; i < 256; ++i) hist[i] = c < 2 ? hh[c * 256 + i] : hh[i] + hh[256 + i];
      GzCode code;
      gz_build_code(hist, &code);
      std::memcpy(ht->lit[c], code.lit, sizeof ht->lit[c]);
      std::memcpy(ht->hdr[c], code.hdr, sizeof ht->hdr[c]);
      for (int i = 0; i < 256; ++i) ht->len3[i] |= (unsigned long long)code.len[i] << (16 * c);
      ht->eob[c] = code.eob;
      ht->hdr_bits[c] = code.hdr_bits;
    }
    gz_crc_table(ht->crc);
    gz_x2n_table(ht->x2n);
    // x^(8 * slice): appends one slice to a CRC; tail[t] = that to the power of the slices behind slice t
    uint32_t step = 1u << 31;
    for (uint64_t nn = kGzSlice, k = 3; nn; nn >>= 1, ++k)
      if (nn & 1u) step = gz_gf_mul(ht->x2n[k & 31u], step);
    uint32_t p = 1u << 31;  // x^0
    for (int t = (int)kGzThreads - 1; t >= 0; --t) {
      ht->tail[t] = p;
      p = gz_gf_mul(step, p);
    }
  }
  CK(cudaMemcpyAsync(e->d_gz_tables.p, ht, sizeof(GzTables), cudaMemcpyHostToDevice, e->st));
  const uint64_t units = (n + kGzUnit - 1) / kGzUnit;
  if (units > 0x7FFFFFFFull) return fail(e, PBSIM_E_INVALID, "stream too large for the gzip writer");
  CK(e->d_gz_usize.ensure((size_t)units * 4 + 64));
  CK(e->d_gz_ucrc.ensure((size_t)units * 4 + 64));
  CK(e->d_gz_usel.ensure((size_t)units * 2 + 64));
  CK(e->d_gz_sbits.ensure((size_t)units * kGzThreads * 2 + 64));
  CK(e->d_gz_uoff.ensure((size_t)(units + 1) * 16 + 64));
  unsigned long long *wide = e->d_gz_uoff.as<unsigned long long>();
  unsigned long long *uoff = wide + (units + 1);
  k_gz_size<<<(uint32_t)units, kGzThreads, 0, e->st>>>(in, n, e->d_gz_tables.as<GzTables>(), bgzf ? 1u : 0u,
                                                     e->d_gz_usize.as<uint32_t>(), e->d_gz_ucrc.as<uint32_t>(),
                                                     e->d_gz_usel.as<uint16_t>(), e->d_gz_sbits.as<uint16_t>());
  CK(cudaMemsetAsync(wide + units, 0, 8, e->st));
  e->launches++;
  const int rc = widen_scan(e, e->d_gz_usize.as<uint32_t>(), (uint32_t)units, wide, uoff);
  if (rc) return rc;
  if (peek(e, hh, uoff + units, 8)) return PBSIM_E_CUDA;
  CK(cudaStreamSynchronize(e->st));
  const uint64_t total = hh[0];
  CK(dst.ensure((size_t)total + 256));
  k_gz_encode<<<(uint32_t)units, kGzThreads, kGzEncodeSmem, e->st>>>(
      in, n, e->d_gz_tables.as<GzTables>(), reinterpret_cast<const uint64_t *>(uoff), e->d_gz_ucrc.as<uint32_t>(),
      e->d_gz_usel.as<uint16_t>(), e->d_gz_sbits.as<uint16_t>(), bgzf ? 1u : 0u, dst.as<uint8_t>());
  e->launches++;
  CK(cudaGetLastError());
  *out_bytes = total;
  return 0;
}

// generate the next batch of the run into output set `set`; 1 = produced, 0 = run finished, < 0 = error
int produce_one(pbsim_engine *e, int set, pbsim_engine::BatchItem *it) {
  for (;;) {
    if (e->len_total >= e->run.len_quota || (e->run.max_reads > 0 && e->reads_done_in_run >= e->run.max_reads)) return 0;
    // batch size: enough reads for the target number of emitted bases, never more than the quota needs
    int64_t nb;
    int64_t clip_room = -1;
    const bool sample = e->model.method == PBSIM_METHOD_SAMPLE;
    SampleBatch sb;
    if (sample) {
      // the groups (pool entry, copies) of the current pool pass that make up this batch (sample_plan.hpp)
      SampleSchedule &S = e->sched;
      sb.skip_first = 0;
      if (!S.pass_open) {
        if (e->run.rng_mode == PBSIM_RNG_REPLAY) {
          const int64_t s0 = e->next_read - e->run.first_read;
          if (s0 >= e->run.replay_nsubreads) return fail(e, PBSIM_E_REPLAY, "replay log exhausted before the quota was reached");
          const int64_t d0 = e->run.replay_starts[s0];
          if (d0 < 0 || d0 >= e->run.replay_ndraws) return fail(e, PBSIM_E_REPLAY, "replay starts are not monotone");
          S.open_pass((int64_t)((uint32_t)e->run.replay_draws[d0] % (uint32_t)S.n));  // sample_value (:1734)
          sb.skip_first = 1;
        } else {
          S.open_pass(SampleSchedule::philox_value(e->run.seed, (uint32_t)e->seq_num, S.pass, (uint32_t)S.n));
        }
      }
      const int64_t target = (e->pipelined && e->mode_to_host) ? std::min(e->target_batch_bases, e->host_batch_bases)
                                                               : e->target_batch_bases;
      const int64_t need = (int64_t)((double)(e->run.len_quota - e->len_total) * 1.05) + (1 << 20);
      int64_t hard = (int64_t)1 << 30;
      if (e->run.rng_mode == PBSIM_RNG_REPLAY) {
        hard = e->run.replay_nsubreads - (e->next_read - e->run.first_read);
        if (hard <= 0) return fail(e, PBSIM_E_REPLAY, "replay log exhausted before the quota was reached");
      }
      sample_collect(S, e->run.batch_reads > 0 ? e->run.batch_reads : (int64_t)1 << 22, std::min(target, need), hard,
                     &e->groups);
      const size_t G = e->groups.entry.size();
      nb = e->groups.first[G];
      if (nb == 0) {  // nothing left in this pass (cannot happen while sample_interval <= n / 2, kept for safety)
        S.next_pass();
        continue;
      }
      CK(e->d_groups.ensure((2 * G + 1) * 4 + 64));
      uint32_t *dg = e->d_groups.as<uint32_t>();
      CK(cudaMemcpyAsync(dg, e->groups.entry.data(), G * 4, cudaMemcpyHostToDevice, e->st));
      CK(cudaMemcpyAsync(dg + G, e->groups.first.data(), (G + 1) * 4, cudaMemcpyHostToDevice, e->st));
      sb.g_entry = dg;
      sb.g_first = dg + G;
      sb.n_groups = (uint32_t)G;
    } else if (e->tail_mode) {
      nb = 1;
      clip_room = e->run.len_quota - e->len_total;
    } else {
      double mean = e->mean_rlen_est > 0 ? e->mean_rlen_est : e->table_mean_len;
      if (e->strategy != PBSIM_STRATEGY_WGS && e->mean_rlen_est <= 0) mean = std::min(mean, e->set_mean_len);
      if (e->strategy == PBSIM_STRATEGY_TEMPL && e->mean_rlen_est <= 0) mean = e->set_mean_len;
      if (mean > (double)e->glen) mean = (double)e->glen;
      if (mean < 1) mean = 1;
      if (e->run.batch_reads > 0) {
        nb = e->run.batch_reads;
      } else {
        int64_t target = (e->pipelined && e->mode_to_host) ? std::min(e->target_batch_bases, e->host_batch_bases)
                                                           : e->target_batch_bases;
        // the first batch of a pipelined run is the only one whose generation nothing hides: keep it short
        if (e->pipelined && e->mode_to_host && e->reads_done_in_run == 0 && e->first_batch_div > 1)
          target = std::max<int64_t>(target / e->first_batch_div, 1 << 26);
        nb = (int64_t)((double)target / (mean * e->model.pass_num));
        nb = std::max<int64_t>(nb, 1 << 12);
        nb = std::min<int64_t>(nb, 1 << 22);
      }
      const double need = (double)(e->run.len_quota - e->len_total) / mean;
      const int64_t est = (int64_t)(need * 1.02) + 16;
      if (est < nb) nb = est;
      if (e->run.max_reads > 0) nb = std::min<int64_t>(nb, e->run.max_reads - e->reads_done_in_run);
      if (e->run.rng_mode == PBSIM_RNG_REPLAY) {
        const int64_t left = e->run.replay_nsubreads / e->model.pass_num - (e->next_read - e->run.first_read);
        if (left <= 0) return fail(e, PBSIM_E_REPLAY, "replay log exhausted before the quota was reached");
        nb = std::min<int64_t>(nb, left);
      }
      if (nb < 1) nb = 1;
    }
    e->cur_set = set;
    CK(cudaEventRecord(e->ev0, e->st));
    BatchResult br;
    int rc = run_batch(e, (uint32_t)nb, clip_room, &br, sample ? &sb : nullptr);
    if (rc) return rc;
    const bool gz = e->deflate && e->mode_to_host && br.n_valid_reads > 0;
    uint64_t gz_bytes[2] = {0, 0};
    if (gz) {
      CK(cudaEventRecord(e->ev_gz[0], e->st));
      // BAM records travel as BGZF blocks (what samtools writes), everything else as plain gzip members
      const bool bgzf = e->bam && e->model.pass_num > 1;
      if ((rc = gz_compress(e, e->out[set].reads.as<uint8_t>(), br.reads_bytes, e->gz[set].reads, &gz_bytes[0], bgzf))) return rc;
      if ((rc = gz_compress(e, e->out[set].maf.as<uint8_t>(), br.maf_bytes, e->gz[set].maf, &gz_bytes[1]))) return rc;
      CK(cudaEventRecord(e->ev_gz[1], e->st));
    }
    CK(cudaEventRecord(e->ev1, e->st));
    CK(cudaStreamSynchronize(e->st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
    e->gen_ms += ms;
    if (getenv("PBSIM_DEBUG")) fprintf(stderr, "[pbsim] batch of %lld reads took %.3f ms on the device\n", (long long)nb, ms);
    if (gz) {
      CK(cudaEventElapsedTime(&ms, e->ev_gz[0], e->ev_gz[1]));
      e->gz_ms += ms;
    }
    const uint32_t pass = (uint32_t)e->model.pass_num;
    const uint32_t nv = br.n_valid_reads;
    if (nv > 0) {
      CK(cudaEventElapsedTime(&ms, e->ev_k[2], e->ev_k[3]));
      e->emit_ms += ms;
    }
    // host-side ordered accumulation of accuracy_total (:2314)
    {
      const double *hacc = reinterpret_cast<const double *>(e->h_acc.p);
      const uint32_t *hrlen = reinterpret_cast<const uint32_t *>(hacc + (size_t)nv * pass);
      uint64_t bases = 0;
      for (uint64_t s = 0; s < (uint64_t)nv * pass; ++s) {
        e->accuracy_total += hacc[s];
        bases += hrlen[s];
      }
      br.bases_all = bases;
    }
    if (sample) {
      if (!br.cut) {
        e->sched.j = e->groups.j_end;
        if (e->sched.j >= e->sched.n) e->sched.next_pass();
      }
    } else if (br.cut) {
      e->tail_mode = true;  // the next read is re-planned with the quota clip, one read at a time
    }
    if (nv == 0) continue;
    if (e->mean_rlen_est <= 0) e->mean_rlen_est = std::max(1.0, (double)br.bases_pass0 / nv);
    it->rc = 1;
    it->set = set;
    it->first_read = e->next_read + 1;
    it->n_reads = nv;
    it->bases = (int64_t)br.bases_all;
    it->reads_text_bytes = br.reads_bytes;
    it->maf_text_bytes = br.maf_bytes;
    it->reads_bytes = gz ? gz_bytes[0] : br.reads_bytes;
    it->maf_bytes = gz ? gz_bytes[1] : br.maf_bytes;
    it->gz = gz;
    e->next_read += nv;
    e->reads_done_in_run += nv;
    e->len_total += (int64_t)br.bases_pass0;
    return 1;
  }
}

// producer thread of the pipeline: fills the output sets alternately, at most one batch ahead of delivery
void producer_main(pbsim_engine *e) {
  cudaSetDevice(e->device);
  for (uint64_t seq = 0;; ++seq) {
    {
      std::unique_lock<std::mutex> lk(e->mu);
      e->cv.wait(lk, [&] { return e->free_sets > 0 || e->stop; });
      if (e->stop) return;
      e->free_sets--;
    }
    pbsim_engine::BatchItem it;
    const int rc = produce_one(e, (int)(seq & 1), &it);
    if (rc != 1) {
      it.rc = rc;
      if (rc < 0) {
        std::lock_guard<std::mutex> lk(e->err_mu);
        it.err = e->err;
      }
    }
    {
      std::lock_guard<std::mutex> lk(e->mu);
      if (rc != 1) e->free_sets++;
      e->queue.push_back(std::move(it));
    }
    e->cv.notify_all();
    if (rc != 1) return;
  }
}

void release_set(pbsim_engine *e) {
  if (!e->pipelined) return;
  {
    std::lock_guard<std::mutex> lk(e->mu);
    e->free_sets++;
  }
  e->cv.notify_all();
}

void stop_producer(pbsim_engine *e) {
  if (e->producer.joinable()) {
    {
      std::lock_guard<std::mutex> lk(e->mu);
      e->stop = true;
    }
    e->cv.notify_all();
    e->producer.join();
  }
  e->queue.clear();
  e->free_sets = 2;
  e->stop = false;
}

// next batch for delivery: 1 = *it is a batch, 0 = finished (or, with block == false, nothing ready yet), < 0 = error
int fetch_batch(pbsim_engine *e, bool block, pbsim_engine::BatchItem *it) {
  if (e->finished) return 0;
  if (!e->pipelined) {
    if (!block) return 0;
    const int rc = produce_one(e, 0, it);
    if (rc == 0) e->finished = true;
    return rc;
  }
  std::unique_lock<std::mutex> lk(e->mu);
  if (block) e->cv.wait(lk, [&] { return !e->queue.empty(); });
  if (e->queue.empty() || (!block && e->queue.front().rc != 1)) return 0;  // end / error surface on a blocking call
  *it = std::move(e->queue.front());
  e->queue.pop_front();
  lk.unlock();
  if (it->rc == 0) e->finished = true;
  if (it->rc < 0) {
    e->finished = true;
    std::lock_guard<std::mutex> g(e->err_mu);
    e->err = it->err;
  }
  return it->rc;
}

// host delivery: start the D2H copy of the next piece into staging slot next_slot
// 1 = a piece is in flight, 0 = nothing to issue (finished, or not ready and !block), < 0 = error
int issue_piece(pbsim_engine *e, bool block) {
  pbsim_engine::Pending &p = e->pend;
  if (!p.active) {
    pbsim_engine::BatchItem it;
    const int rc = fetch_batch(e, block, &it);
    if (rc != 1) return rc;
    p = pbsim_engine::Pending();
    p.active = true;
    p.set = it.set;
    p.gz = it.gz;
    p.text[0] = it.reads_text_bytes;
    p.text[1] = it.maf_text_bytes;
    p.total[0] = it.reads_bytes;
    p.total[1] = it.maf_bytes;
    p.first_read = it.first_read;
    p.n_reads = it.n_reads;
    p.bases = it.bases;
  }
  for (int k = 0; k < 2; ++k)
    for (int slot = 0; slot < 2; ++slot) CK(e->h_stage[k][slot].ensure(e->stage_bytes));
  const pbsim_engine::OutSet &O = p.gz ? e->gz[p.set] : e->out[p.set];
  const uint8_t *src[2] = {O.reads.as<uint8_t>(), O.maf.as<uint8_t>()};
  pbsim_engine::Piece &q = e->piece;
  q = pbsim_engine::Piece();
  q.valid = true;
  q.slot = e->next_slot;
  for (int k = 0; k < 2; ++k) {
    const uint64_t n = std::min<uint64_t>(e->stage_bytes, p.total[k] - p.issued[k]);
    q.bytes[k] = n;
    if (n) CK(cudaMemcpyAsync(e->h_stage[k][q.slot].p, src[k] + p.issued[k], n, cudaMemcpyDeviceToHost, e->st_copy));
    p.issued[k] += n;
  }
  CK(cudaEventRecord(e->ev_copy, e->st_copy));
  if (p.first) {
    q.first = true;
    q.text[0] = p.text[0];
    q.text[1] = p.text[1];
    q.first_read = p.first_read;
    q.n_reads = p.n_reads;
    q.bases = p.bases;
    p.first = false;
  }
  if (p.issued[0] >= p.total[0] && p.issued[1] >= p.total[1]) {
    q.release_set = p.set;
    p.active = false;
  }
  e->next_slot ^= 1;
  return 1;
}

int next_chunk_impl(pbsim_engine *e, pbsim_chunk *c, bool to_host) {
  if (!e || !c) return PBSIM_E_INVALID;
  if (!e->running) return fail(e, PBSIM_E_INVALID, "simulate_begin was not called");
  std::memset(c, 0, sizeof *c);
  if (!e->mode_set) {
    e->mode_set = true;
    e->mode_to_host = to_host;
    e->pipelined = e->pipeline == 2 || (e->pipeline == 1 && to_host);
    if (e->pipelined) e->producer = std::thread(producer_main, e);
  } else if (e->mode_to_host != to_host) {
    return fail(e, PBSIM_E_INVALID, "host and device delivery cannot be mixed within one run");
  }
  if (to_host) {
    if (!e->piece.valid) {
      const int rc = issue_piece(e, true);
      if (rc != 1) return rc;
    }
    pbsim_engine::Piece q = e->piece;
    CK(cudaEventSynchronize(e->ev_copy));
    e->piece.valid = false;
    if (q.release_set >= 0) release_set(e);  // the batch has left HBM: the producer may overwrite its set
    c->reads = reinterpret_cast<const char *>(e->h_stage[0][q.slot].p);
    c->reads_bytes = (int64_t)q.bytes[0];
    c->maf = reinterpret_cast<const char *>(e->h_stage[1][q.slot].p);
    c->maf_bytes = (int64_t)q.bytes[1];
    c->on_device = 0;
    c->compressed = e->deflate ? 1 : 0;
    if (q.first) {
      c->first_read = q.first_read;
      c->n_reads = q.n_reads;
      c->bases = q.bases;
      c->reads_text_bytes = (int64_t)q.text[0];
      c->maf_text_bytes = (int64_t)q.text[1];
    }
    // prefetch the next piece into the other slot while the caller consumes this one
    const int rc = issue_piece(e, false);
    if (rc < 0) return rc;
    return 1;
  }
  if (e->held_set >= 0) {  // the caller is done with the previous device chunk
    release_set(e);
    e->held_set = -1;
  }
  pbsim_engine::BatchItem it;
  const int rc = fetch_batch(e, true, &it);
  if (rc != 1) return rc;
  e->held_set = it.set;
  c->first_read = it.first_read;
  c->n_reads = it.n_reads;
  c->bases = it.bases;
  c->reads_bytes = (int64_t)it.reads_bytes;
  c->maf_bytes = (int64_t)it.maf_bytes;
  c->reads_text_bytes = (int64_t)it.reads_text_bytes;
  c->maf_text_bytes = (int64_t)it.maf_text_bytes;
  c->reads = reinterpret_cast<const char *>(e->out[it.set].reads.p);
  c->maf = reinterpret_cast<const char *>(e->out[it.set].maf.p);
  c->on_device = 1;
  return 1;
}

// Replay of simulate_by_errhmm_trans: the reference copies an accuracy-100 read with `for (i=0; i<mut.len; i++)`
// (pbsim.cpp:4532) using the SAME i that counts the transcript's reads (:4487), so after such a read the count
// continues from mut.len + 1 and the transcript's remaining reads are (usually) never simulated.  Which reads exist
// therefore depends on the draws.  The log holds them: walk it with the planner's three draws per read (:4538-4562)
// and record the transcript and the rank of every logged read.
int build_replay_read_map(pbsim_engine *e) {
  const pbsim_run &run = e->run;
  const int64_t pass = e->model.pass_num;
  const int64_t n_logged = run.replay_nsubreads / pass;
  std::vector<uint32_t> map_tr, map_k;
  map_tr.reserve((size_t)n_logged);
  map_k.reserve((size_t)n_logged);
  int64_t idx = 0;
  for (uint32_t t = 0; t < (uint32_t)e->set_n && idx < n_logged; ++t) {
    const uint32_t tlen = e->h_set_start[t + 1] - e->h_set_start[t];
    const uint32_t rank = (tlen + 999u) / 1000u;
    for (uint64_t k = 1; k <= e->h_set_nr[t] && idx < n_logged; ++k) {
      const int64_t st = run.replay_starts[idx * pass];
      if (st < 0 || st + 3 > run.replay_ndraws) return fail(e, PBSIM_E_REPLAY, "replay log exhausted while mapping the reads of the set");
      const uint32_t d0 = (uint32_t)run.replay_draws[st], d1 = (uint32_t)run.replay_draws[st + 1],
                     d2 = (uint32_t)run.replay_draws[st + 2];
      uint32_t len = (uint32_t)e->h_prob2len[d0 % (uint32_t)e->model.len_rand_value];
      const uint32_t acc = e->h_prob2acc[d1 % (uint32_t)e->model.accuracy_rand_value];
      const uint32_t index = d2 % e->h_ssp_mod[rank] + 1u;
      uint32_t ssp = 100u;
      for (uint32_t j = 0; j < 21u; ++j) {
        const uint32_t en = e->h_ssp_ends[rank * 21u + j];
        if (en == 0xFFFFu) break;
        if (index <= en) {
          ssp = j * 5u;
          break;
        }
      }
      const double value = ssp == 0u ? 0.0 : ((double)ssp - 2.5) / 100;
      volatile double prod = (double)tlen * value;  // two roundings, as plan_read_trans computes it
      const uint32_t offset = (uint32_t)(int)(prod + 0.5);
      if ((uint64_t)offset + len > tlen) len = offset < tlen ? tlen - offset : 0u;
      map_tr.push_back(t);
      map_k.push_back((uint32_t)k);
      ++idx;
      if (acc == 100u) k = len;  // the loop variable was the copy loop's too: the count resumes behind mut.len
    }
  }
  if (idx != n_logged)
    return fail(e, PBSIM_E_REPLAY, "the replay log holds %lld reads but the set accounts for %lld", (long long)n_logged,
                (long long)idx);
  int rc;
  if ((rc = upload(e, e->d_map_tr, map_tr.data(), map_tr.size()))) return rc;
  if ((rc = upload(e, e->d_map_k, map_k.data(), map_k.size()))) return rc;
  CK(cudaStreamSynchronize(e->st));
  e->replay_map = true;
  e->run.max_reads = idx;
  return 0;
}

}  // namespace

extern "C" {

int pbsim_cuda_abi_version(void) { return PBSIM_ABI_VERSION; }

const char *pbsim_cuda_last_error(const pbsim_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int pbsim_cuda_create(pbsim_engine **out, int device) {
  pbsim_engine *e = nullptr;
  if (!out) return fail(e, PBSIM_E_INVALID, "null output pointer");
  int n = 0;
  cudaError_t ce = cudaGetDeviceCount(&n);
  if (ce != cudaSuccess || n == 0)
    return fail(e, PBSIM_E_CUDA, "no usable CUDA device (%s); libpbsim_cuda has no CPU fallback",
                ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
  if (device < 0 || device >= n) return fail(e, PBSIM_E_INVALID, "device %d out of range (0..%d)", device, n - 1);
  CK(cudaSetDevice(device));
  // Function attributes belong to the function as loaded on one device, so every engine sets them on its own.
  // k_emit_rows' staging rows need shared memory for 4 CTAs per SM; k_qs_pass1 gets the largest carve-out too.
  CK(cudaFuncSetAttribute(k_qs_pass1, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CK(cudaFuncSetAttribute(k_emit_rows<PBSIM_METHOD_QSHMM>, cudaFuncAttributePreferredSharedMemoryCarveout,
                          cudaSharedmemCarveoutMaxShared));
  CK(cudaFuncSetAttribute(k_emit_rows<PBSIM_METHOD_ERRHMM>, cudaFuncAttributePreferredSharedMemoryCarveout,
                          cudaSharedmemCarveoutMaxShared));
  CK(cudaFuncSetAttribute(k_gz_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGzEncodeSmem));
  pbsim_engine *ne = new pbsim_engine();
  ne->device = device;
  cudaError_t c1 = cudaStreamCreateWithFlags(&ne->st, cudaStreamNonBlocking);
  cudaError_t c2 = cudaStreamCreateWithFlags(&ne->st_copy, cudaStreamNonBlocking);
  cudaError_t c3 = cudaEventCreate(&ne->ev0);
  cudaError_t c4 = cudaEventCreate(&ne->ev1);
  if (c1 != cudaSuccess || c2 != cudaSuccess || c3 != cudaSuccess || c4 != cudaSuccess) {
    delete ne;
    return fail(e, PBSIM_E_CUDA, "cannot create CUDA streams/events");
  }
  cudaEventCreate(&ne->ev_copy);
  for (auto &ev : ne->ev_k) cudaEventCreate(&ev);
  for (auto &ev : ne->ev_user) cudaEventCreate(&ev);
  for (auto &ev : ne->ev_gz) cudaEventCreate(&ev);
  for (auto &ev : ne->ev_seg) cudaEventCreate(&ev);
  for (auto &ev : ne->ev_chain) cudaEventCreate(&ev);
  std::memset(&ne->model, 0, sizeof ne->model);
  std::memset(&ne->emitp, 0, sizeof ne->emitp);
  *out = ne;
  return 0;
}

void pbsim_cuda_destroy(pbsim_engine *e) {
  if (!e) return;
  cudaSetDevice(e->device);
  stop_producer(e);
  cudaStreamSynchronize(e->st_copy);
  cudaStreamSynchronize(e->st);
  cudaEventDestroy(e->ev_copy);
  for (auto &ev : e->ev_k) cudaEventDestroy(ev);
  for (auto &ev : e->ev_user) cudaEventDestroy(ev);
  for (auto &ev : e->ev_gz) cudaEventDestroy(ev);
  for (auto &ev : e->ev_seg) cudaEventDestroy(ev);
  for (auto &ev : e->ev_chain) cudaEventDestroy(ev);
  cudaEventDestroy(e->ev0);
  cudaEventDestroy(e->ev1);
  cudaStreamDestroy(e->st);
  cudaStreamDestroy(e->st_copy);
  delete e;  // the buffers free themselves, on the engine's device
}

int pbsim_cuda_set_model(pbsim_engine *e, const pbsim_model *m) {
  if (!e || !m) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  const bool sample = m->method == PBSIM_METHOD_SAMPLE;
  if (m->method != PBSIM_METHOD_QSHMM && m->method != PBSIM_METHOD_ERRHMM && !sample)
    return fail(e, PBSIM_E_INVALID, "method must be qshmm, errhmm or sample");
  if (sample && m->pass_num != 1)
    return fail(e, PBSIM_E_INVALID, "sampling-based simulation supports only single-pass");  // pbsim.cpp:1675-1679
  if (!sample &&
      (m->pass_num < 1 || m->len_rand_value < 1 || m->accuracy_rand_value < 1 || !m->prob2len || !m->prob2accuracy))
    return fail(e, PBSIM_E_INVALID, "model samplers are empty");
  if (m->len_max > 1000000) return fail(e, PBSIM_E_INVALID, "length-max above FASTQ_LEN_MAX (1000000)");
  if (!e->img.build(*m)) return fail(e, PBSIM_E_INVALID, "model tables: %s", e->img.error.c_str());
  e->model = *m;
  if (sample) {  // lengths come from the pool (set_pool); there are no samplers
    e->h_prob2len.assign(1, 0);
    e->h_prob2acc.assign(1, 0);
    e->model.len_rand_value = e->model.accuracy_rand_value = 1;
  } else {
    e->h_prob2len.assign(m->prob2len, m->prob2len + m->len_rand_value);
    e->h_prob2acc.assign(m->prob2accuracy, m->prob2accuracy + m->accuracy_rand_value);
  }
  {
    double acc = 0;
    for (int32_t v : e->h_prob2len) acc += v;
    e->table_mean_len = acc / e->h_prob2len.size();
  }
  e->model.prob2len = e->h_prob2len.data();
  e->model.prob2accuracy = e->h_prob2acc.data();
  // NOTE: e->model.rows[] still points into the caller's tables; apply_bias reads emis_del from them,
  // so the caller keeps the pbsim_model alive while the engine uses it (documented in the header).
  if (upload(e, e->d_blob, e->img.blob.data(), e->img.blob.size())) return PBSIM_E_CUDA;
  if (upload(e, e->d_acc, e->img.acc, PBSIM_NACC)) return PBSIM_E_CUDA;
  if (upload(e, e->d_prob2len, e->h_prob2len.data(), e->h_prob2len.size())) return PBSIM_E_CUDA;
  if (upload(e, e->d_prob2acc, e->h_prob2acc.data(), e->h_prob2acc.size())) return PBSIM_E_CUDA;
  CK(e->d_qs_tabs.ensure(kQsTabBytes));
  CK(e->d_qs_thr_hp.ensure(PBSIM_NQV * 48));
  CK(e->d_qs_thr_hp32.ensure(PBSIM_NQV * 48));
  CK(e->d_er_bias.ensure(std::max<size_t>(e->img.er_bias.size() * 2, 16) + 64));
  // errhmm: largest per-accuracy shared-memory footprint
  e->er_smem_bar_off = 0;
  if (m->method == PBSIM_METHOD_ERRHMM) {
    uint32_t mx = 0;
    for (int a = 0; a < PBSIM_NACC; ++a) {
      const AccEntry &ae = e->img.acc[a];
      if (!ae.valid || ae.mode == 3) continue;
      const uint32_t need = ae.blob_bytes + ((ae.nstates + 1u) * 2u + 15u) / 16u * 16u;
      mx = std::max(mx, need);
    }
    e->er_smem_bar_off = (mx + 15u) / 16u * 16u;
    const int smem = (int)e->er_smem_bar_off + 16;
    CK(cudaFuncSetAttribute(k_sim_errhmm<PBSIM_RNG_PHILOX>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CK(cudaFuncSetAttribute(k_sim_errhmm<PBSIM_RNG_REPLAY>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CK(cudaFuncSetAttribute(k_sim_seg_err, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CK(cudaFuncSetAttribute(k_chain_chunk_err, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  // emission constants
  e->emitp.pass_num = (uint32_t)m->pass_num;
  e->emitp.sam = m->pass_num > 1 ? 1u : 0u;
  snprintf(e->emitp.rq, sizeof e->emitp.rq, "%f", m->accuracy_mean);
  e->emitp.rq_len = (uint32_t)strlen(e->emitp.rq);
  e->emitp.rq_f = strtof(e->emitp.rq, nullptr);  // what a SAM parser makes of "rq:f:0.850000"
  // stats block
  e->freq_len_cells = 2 * m->len_max + 2;
  e->stats_cells = kStatCounters + 100001 + e->freq_len_cells;
  CK(e->d_stats.ensure((size_t)e->stats_cells * 8));
  CK(cudaStreamSynchronize(e->st));
  e->model_set = true;
  if (e->seq_set) return upload_bias_tables(e);
  return 0;
}

int pbsim_cuda_set_pool(pbsim_engine *e, const char *quals, const int64_t *qstart, int64_t n) {
  if (!e || !quals || !qstart) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (e->running) return fail(e, PBSIM_E_INVALID, "the pool cannot change during a run");
  if (n < 2) return fail(e, PBSIM_E_INVALID, "the pool needs at least 2 reads (the reference divides by zero, pbsim.cpp:1723)");
  if (n > 0xFFFFFFF0ll) return fail(e, PBSIM_E_INVALID, "too many reads in the pool");
  if (qstart[0] != 0) return fail(e, PBSIM_E_INVALID, "qstart[0] must be 0");
  for (int64_t j = 0; j < n; ++j) {
    const int64_t len = qstart[j + 1] - qstart[j];
    if (len < 1 || len > 1000000)  // FASTQ_LEN_MAX :27
      return fail(e, PBSIM_E_INVALID, "pool read %lld has %lld qualities (1..1000000)", (long long)j + 1, (long long)len);
  }
  const int64_t total = qstart[n];
  for (int64_t i = 0; i < total; ++i)
    if ((uint8_t)quals[i] < 33 || (uint8_t)quals[i] > 126)
      return fail(e, PBSIM_E_INVALID, "quality character out of range '!'..'~' at pool byte %lld", (long long)i);
  e->pool_start.assign(qstart, qstart + n + 1);
  int rc;
  if ((rc = upload(e, e->d_pool_q, reinterpret_cast<const uint8_t *>(quals), (size_t)total))) return rc;
  if ((rc = upload(e, e->d_pool_start, reinterpret_cast<const uint64_t *>(e->pool_start.data()), (size_t)n + 1))) return rc;
  CK(cudaStreamSynchronize(e->st));
  e->pool_set = true;
  return 0;
}

int pbsim_cuda_set_sequence(pbsim_engine *e, const pbsim_sequence *s) {
  if (!e || !s || !s->bases) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (s->len < 1 || s->len > 1000000000) return fail(e, PBSIM_E_INVALID, "sequence length out of range");
  const int rc = upload_ascii(e, s->bases, s->len);
  if (rc) return rc;
  e->strategy = PBSIM_STRATEGY_WGS;
  e->seq_name.clear();
  return finish_sequence_ingest(e, s->len, s->seq_num, s->hp_del_bias);
}

int pbsim_cuda_set_sequence_name(pbsim_engine *e, const char *name) {
  if (!e || !name) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  const size_t n = strlen(name);
  if (n < 1 || n > 4096) return fail(e, PBSIM_E_INVALID, "sequence name must have 1 to 4096 characters");
  for (size_t i = 0; i < n; ++i)
    if ((unsigned char)name[i] <= ' ' || (unsigned char)name[i] > '~')
      return fail(e, PBSIM_E_INVALID, "sequence name must be printable characters without whitespace");
  if (e->running) return fail(e, PBSIM_E_INVALID, "the sequence name cannot change during a run");
  CK(e->d_rname.ensure(n + 16));
  CK(cudaMemcpy(e->d_rname.p, name, n, cudaMemcpyHostToDevice));
  e->seq_name.assign(name, n);
  return 0;
}

int pbsim_cuda_set_seqset(pbsim_engine *e, const pbsim_seqset *s) {
  if (!e || !s || !s->bases || !s->start || !s->ids || !s->id_start) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (!e->model_set) return fail(e, PBSIM_E_INVALID, "set_model must precede set_seqset");
  if (s->strategy != PBSIM_STRATEGY_TRANS && s->strategy != PBSIM_STRATEGY_TEMPL)
    return fail(e, PBSIM_E_INVALID, "seqset strategy must be PBSIM_STRATEGY_TRANS or PBSIM_STRATEGY_TEMPL");
  const bool trans = s->strategy == PBSIM_STRATEGY_TRANS;
  if (trans && (!s->plus_exp || !s->minus_exp)) return fail(e, PBSIM_E_INVALID, "transcripts need plus_exp and minus_exp");
  if (s->n < 1 || s->n > 100000000) return fail(e, PBSIM_E_INVALID, "number of sequences out of range");
  const int64_t total = s->start[s->n];
  if (s->start[0] != 0 || total < 1 || total > 0xFFFF0000ll)
    return fail(e, PBSIM_E_INVALID, "sequence set too large for one engine (%lld bases; limit 2^32 - 2^16)", (long long)total);
  const uint32_t n = (uint32_t)s->n;
  std::vector<uint32_t> start(n + 1), plus_w(2 * (size_t)n, 0u), idst(n + 1);
  std::vector<uint64_t> rprefix(n + 1);
  int64_t max_len = 0;
  uint64_t reads = 0;
  for (uint32_t t = 0; t < n; ++t) {
    const int64_t len = s->start[t + 1] - s->start[t];
    if (len < 0) return fail(e, PBSIM_E_INVALID, "start[] must not decrease");
    // TEMPLATE_LEN_MAX :29; transcripts: prob2ssp has TR_RANK_MAX = 1000 rows, rank = ceil(len / 1000) (:44, :2507)
    if (len > (trans ? 999000 : 1000000))
      return fail(e, PBSIM_E_INVALID, "sequence %u is too long (%lld bases)", t + 1, (long long)len);
    uint64_t nr = 1;
    if (trans) {
      if (s->plus_exp[t] < 0 || s->minus_exp[t] < 0) return fail(e, PBSIM_E_INVALID, "negative expression value");
      nr = (uint64_t)s->plus_exp[t] + (uint64_t)s->minus_exp[t];
      plus_w[t] = (uint32_t)s->plus_exp[t];
      plus_w[n + t] = (uint32_t)nr;  // weight of the sequence in the --hp-del-bias prepass (:2714)
    }
    // a window can be empty when a start fraction of 97.5 % meets a transcript of <= 20 bases (:2860-2866); the
    // reference then divides by zero and indexes freq_accuracy with the result: undefined there, refused here
    if (nr > 0 && len < (trans ? 21 : 1))
      return fail(e, PBSIM_E_INVALID, "sequence %u has %lld bases: %s", t + 1, (long long)len,
                  trans ? "transcripts that are read must be longer than 20 bases" : "empty template");
    start[t] = (uint32_t)s->start[t];
    idst[t] = (uint32_t)s->id_start[t];
    if (s->id_start[t + 1] < s->id_start[t] || s->id_start[t + 1] - s->id_start[t] > 128)
      return fail(e, PBSIM_E_INVALID, "name of sequence %u is longer than 128 characters", t + 1);
    rprefix[t] = reads;
    reads += nr;
    max_len = std::max(max_len, len);
  }
  start[n] = (uint32_t)total;
  idst[n] = (uint32_t)s->id_start[n];
  rprefix[n] = reads;
  if (reads < 1) return fail(e, PBSIM_E_INVALID, "the set yields no reads");
  if (reads > 0xFFFFFFF0ull) return fail(e, PBSIM_E_INVALID, "too many reads for one run");
  e->strategy = s->strategy;
  e->set_n = n;
  e->set_total_reads = (int64_t)reads;
  e->h_set_start = start;
  e->h_set_nr.assign(n, 1u);
  if (trans)
    for (uint32_t t = 0; t < n; ++t) e->h_set_nr[t] = plus_w[n + t];
  e->set_mean_len = (double)total / n;
  int rc;
  if ((rc = upload(e, e->d_set_start, start.data(), start.size()))) return rc;
  if ((rc = upload(e, e->d_set_rprefix, rprefix.data(), rprefix.size()))) return rc;
  if ((rc = upload(e, e->d_set_plus, plus_w.data(), plus_w.size()))) return rc;
  if ((rc = upload(e, e->d_set_idstart, idst.data(), idst.size()))) return rc;
  if ((rc = upload(e, e->d_set_ids, reinterpret_cast<const uint8_t *>(s->ids), (size_t)idst[n]))) return rc;
  if (trans) {
    e->set_rank_max = (int32_t)std::ceil((float)max_len / 1000);  // transcript.rank_max (:1137)
    std::vector<uint16_t> ends((size_t)(e->set_rank_max + 1) * 21), mod((size_t)e->set_rank_max + 1);
    pbsim_host_ssp_table(e->set_rank_max, ends.data(), mod.data());
    e->h_ssp_ends = ends;
    e->h_ssp_mod = mod;
    if ((rc = upload(e, e->d_set_ssp_ends, ends.data(), ends.size()))) return rc;
    if ((rc = upload(e, e->d_set_ssp_mod, mod.data(), mod.size()))) return rc;
    CK(cudaStreamSynchronize(e->st));  // the vectors go out of scope
  }
  if ((rc = upload_ascii(e, s->bases, total))) return rc;
  // only simulate_by_qshmm_trans upper-cases the first base (:2774; :3330, :4474, :5049 start at 1)
  const bool keep_first = !(trans && e->model.method == PBSIM_METHOD_QSHMM);
  rc = finish_sequence_ingest(e, total, 0, s->hp_del_bias, keep_first);
  return rc;
}

int pbsim_cuda_set_synthetic_sequence(pbsim_engine *e, int64_t len, int32_t seq_num, uint64_t seed) {
  if (!e) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (len < 1 || len > 1000000000) return fail(e, PBSIM_E_INVALID, "sequence length out of range");
  const int rc = upload_ascii(e, nullptr, len);
  if (rc) return rc;
  k_synth_ascii<<<nblk((len + 15) / 16, 256), 256, 0, e->st>>>(e->d_ascii.as<uint8_t>(), len, seed);
  e->launches++;
  double bias[12] = {0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0};
  e->strategy = PBSIM_STRATEGY_WGS;
  e->seq_name.clear();
  return finish_sequence_ingest(e, len, seq_num, bias);
}

int pbsim_cuda_update_hp_del_bias(pbsim_engine *e, const double bias[12]) {
  if (!e || !bias || !e->seq_set) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  for (int h = 1; h <= 11; ++h)
    if ((bias[h] == 1.0) != (e->bias[h] == 1.0))
      return fail(e, PBSIM_E_INVALID, "update_hp_del_bias may only change values, not which cells equal 1; call set_sequence");
  std::memcpy(e->bias, bias, sizeof e->bias);
  if (e->model_set) return upload_bias_tables(e);
  return 0;
}

int pbsim_cuda_get_sequence_ascii(pbsim_engine *e, char *dst, int64_t cap) {
  if (!e || !dst || !e->seq_set || cap < e->glen) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  CK(cudaMemcpyAsync(dst, e->d_ascii.p, (size_t)e->glen, cudaMemcpyDeviceToHost, e->st));
  CK(cudaStreamSynchronize(e->st));
  return 0;
}

int pbsim_cuda_get_hpfreq(pbsim_engine *e, int64_t hpfreq[12]) {
  if (!e || !e->seq_set) return PBSIM_E_INVALID;
  std::memcpy(hpfreq, e->hpfreq, sizeof e->hpfreq);
  return 0;
}

int pbsim_cuda_simulate_begin(pbsim_engine *e, const pbsim_run *run) {
  if (!e || !run) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (!e->model_set || !e->seq_set) return fail(e, PBSIM_E_INVALID, "set_model and set_sequence must precede simulate_begin");
  if (run->rng_mode == PBSIM_RNG_REPLAY && (!run->replay_draws || !run->replay_starts || run->replay_nsubreads < 1))
    return fail(e, PBSIM_E_INVALID, "replay mode needs the draw log and the subread starts");
  if (e->align && e->bam) return fail(e, PBSIM_E_INVALID, "options align and bam cannot be combined (alignment lines are SAM text)");
  if (e->align && e->strategy == PBSIM_STRATEGY_WGS && e->seq_name.empty())
    return fail(e, PBSIM_E_INVALID, "option align needs pbsim_cuda_set_sequence_name after set_sequence (the RNAME of the records)");
  // a run abandoned without simulate_end: its producer thread must be gone before any run state changes
  stop_producer(e);
  CK(cudaStreamSynchronize(e->st_copy));  // a piece of that run may still be on its way into the staging buffers
  e->running = false;
  if (e->model.method == PBSIM_METHOD_SAMPLE) {
    if (!e->pool_set) return fail(e, PBSIM_E_INVALID, "set_pool must precede simulate_begin for --method sample");
    if (e->strategy != PBSIM_STRATEGY_WGS) return fail(e, PBSIM_E_INVALID, "--method sample simulates a genome (--strategy wgs)");
    if (run->first_read != 0 || run->len_total_start != 0 || run->max_reads != 0)
      return fail(e, PBSIM_E_INVALID, "--method sample runs whole sequences: read ranges are not supported");
    if (!e->sched.init(run->len_quota, (int64_t)e->pool_start.size() - 1, e->pool_start.data()))
      return fail(e, PBSIM_E_INVALID, "the pool cannot be sampled (fewer than 2 reads)");
    e->sample_spec_run = true;
    e->sample_redo_groups = 0;
  }
  e->run = *run;
  e->replay_map = false;
  if (e->strategy != PBSIM_STRATEGY_WGS) {
    // the whole set (or the requested range of its read numbers) is the run; there is no quota (:2841, :3312)
    if (run->first_read < 0 || run->first_read >= e->set_total_reads)
      return fail(e, PBSIM_E_INVALID, "first_read is outside the set's %lld reads", (long long)e->set_total_reads);
    const int64_t left = e->set_total_reads - run->first_read;
    e->run.len_quota = INT64_MAX / 4;
    e->run.len_total_start = 0;
    e->run.max_reads = run->max_reads > 0 ? std::min(run->max_reads, left) : left;
    if (run->rng_mode == PBSIM_RNG_REPLAY && e->strategy == PBSIM_STRATEGY_TRANS && e->model.method == PBSIM_METHOD_ERRHMM) {
      if (run->first_read != 0)
        return fail(e, PBSIM_E_INVALID, "a replay of simulate_by_errhmm_trans starts at read 0 (its read numbering depends on the draws)");
      const int rc = build_replay_read_map(e);
      if (rc) return rc;
    }
  }
  e->next_read = run->first_read;
  e->len_total = e->run.len_total_start;
  e->reads_done_in_run = 0;
  e->finished = false;
  e->tail_mode = false;
  e->mean_rlen_est = 0;
  e->accuracy_total = 0;
  e->gen_ms = 0;
  e->sim_ms = 0;
  e->emit_ms = 0;
  e->gz_ms = 0;
  e->seg_ms = 0;
  e->chain_ms = 0;
  e->pend = pbsim_engine::Pending();
  e->piece = pbsim_engine::Piece();
  e->next_slot = 0;
  e->held_set = -1;
  e->mode_set = false;
  e->pipelined = false;
  e->launches = 0;
  k_init_stats<<<nblk(e->stats_cells, 256), 256, 0, e->st>>>(e->d_stats.as<unsigned long long>(), e->stats_cells);
  e->launches++;
  CK(cudaGetLastError());
  e->running = true;
  return 0;
}

int pbsim_cuda_next_chunk(pbsim_engine *e, pbsim_chunk *c) {
  if (e) cudaSetDevice(e->device);
  return next_chunk_impl(e, c, true);
}

int pbsim_cuda_next_chunk_device(pbsim_engine *e, pbsim_chunk *c) {
  if (e) cudaSetDevice(e->device);
  return next_chunk_impl(e, c, false);
}

int pbsim_cuda_simulate_end(pbsim_engine *e, pbsim_stats *st, int64_t *freq_len, int64_t freq_len_cells,
                            int64_t *freq_accuracy) {
  if (!e || !st) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (!e->running) return fail(e, PBSIM_E_INVALID, "simulate_begin was not called");
  stop_producer(e);
  CK(cudaStreamSynchronize(e->st_copy));
  // The block is 16 + 100001 + 2 len_max + 2 cells (16.8 MB with --length-max 1000000) and the GPU idles while the host
  // looks at it: fetch the counters and the accuracy histogram into pinned memory first, then only the occupied range
  // [res_len_min, res_len_max] of the length histogram.
  CK(e->h_stats.ensure((size_t)e->stats_cells * 8));
  long long *blk = reinterpret_cast<long long *>(e->h_stats.p);
  const size_t head_cells = (size_t)kStatCounters + 100001;
  CK(cudaMemcpyAsync(blk, e->d_stats.p, head_cells * 8, cudaMemcpyDeviceToHost, e->st));
  CK(cudaStreamSynchronize(e->st));
  std::memset(st, 0, sizeof *st);
  st->res_num = blk[0];
  st->res_pass_num = blk[1];
  st->res_len_total = blk[2];
  st->res_len_min = blk[3];
  st->res_len_max = blk[4];
  st->res_sub_num = blk[5];
  st->res_ins_num = blk[6];
  st->res_del_num = blk[7];
  st->accuracy_total = e->accuracy_total;
  const long long *fa = blk + kStatCounters;
  long long *fl = blk + head_cells;
  int64_t fl_lo = 0, fl_hi = 0;  // occupied cells of freq_len: [fl_lo, fl_hi)
  if (st->res_pass_num > 0) {
    fl_lo = std::min<int64_t>(std::max<int64_t>(st->res_len_min, 0), e->freq_len_cells);
    fl_hi = std::min<int64_t>(std::max<int64_t>(st->res_len_max + 1, fl_lo), e->freq_len_cells);
    if (fl_hi > fl_lo) {
      CK(cudaMemcpyAsync(fl + fl_lo, reinterpret_cast<const long long *>(e->d_stats.p) + head_cells + fl_lo,
                         (size_t)(fl_hi - fl_lo) * 8, cudaMemcpyDeviceToHost, e->st));
      CK(cudaStreamSynchronize(e->st));
    }
  }
  // mean / SD exactly as the reference derives them from the histograms (:2387-2410); cells outside the occupied range
  // are zero and add nothing
  if (st->res_pass_num > 0) {
    st->res_len_mean = (double)st->res_len_total / st->res_pass_num;
    st->res_accuracy_mean = e->accuracy_total / st->res_pass_num;
    if (st->res_pass_num == 1) {
      st->res_len_sd = 0.0;
      st->res_accuracy_sd = 0.0;
    } else {
      double variance = 0.0;
      for (int64_t i = fl_lo; i <= e->model.len_max && i < fl_hi; ++i)
        if (fl[i] > 0) variance += pow((st->res_len_mean - i), 2) * fl[i];
      st->res_len_sd = sqrt(variance / st->res_pass_num);
      variance = 0.0;
      for (int64_t i = 0; i <= 100000; ++i)
        if (fa[i] > 0) variance += pow((st->res_accuracy_mean - i * 0.00001), 2) * fa[i];
      st->res_accuracy_sd = sqrt(variance / st->res_pass_num);
    }
  }
  st->gen_seconds = e->gen_ms * 1e-3;
  st->sim_seconds = e->sim_ms * 1e-3;
  st->emit_seconds = e->emit_ms * 1e-3;
  st->deflate_seconds = e->gz_ms * 1e-3;
  st->seg_seconds = e->seg_ms * 1e-3;
  st->chain_seconds = e->chain_ms * 1e-3;
  st->kernel_launches = e->launches;
  st->len_total_end = e->len_total;
  if (freq_len) {
    const int64_t n = std::min<int64_t>(freq_len_cells, e->freq_len_cells);
    for (int64_t i = 0; i < n; ++i) freq_len[i] = (i >= fl_lo && i < fl_hi) ? fl[i] : 0;
  }
  if (freq_accuracy)
    for (int64_t i = 0; i <= 100000; ++i) freq_accuracy[i] = fa[i];
  e->running = false;
  return 0;
}

int pbsim_cuda_device_timer(pbsim_engine *e, int stop, double *ms) {
  if (!e) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (!stop) {
    CK(cudaStreamSynchronize(e->st));
    CK(cudaEventRecord(e->ev_user[0], e->st));
    return 0;
  }
  CK(cudaEventRecord(e->ev_user[1], e->st));
  CK(cudaEventSynchronize(e->ev_user[1]));
  float f = 0;
  CK(cudaEventElapsedTime(&f, e->ev_user[0], e->ev_user[1]));
  if (ms) *ms = f;
  return 0;
}

int pbsim_cuda_set_option(pbsim_engine *e, const char *name, int64_t value) {
  if (!e || !name) return PBSIM_E_INVALID;
  if (!strcmp(name, "stage_bytes")) {
    if (value < 4096) return fail(e, PBSIM_E_INVALID, "stage_bytes too small");
    if (e->pend.active || e->piece.valid) return fail(e, PBSIM_E_INVALID, "cannot resize staging while pieces are pending");
    e->stage_bytes = (size_t)value;
    for (auto &a : e->h_stage)
      for (auto &b : a) b.release();
    return 0;
  }
  if (!strcmp(name, "segments")) {
    e->seg_enabled = value != 0;
    return 0;
  }
  if (!strcmp(name, "chain_chunk")) {
    if (value < 0 || value > 65536) return fail(e, PBSIM_E_INVALID, "chain_chunk must be 0 (by method) or 1..65536 segments");
    e->chain_chunk = value;
    return 0;
  }
  if (!strcmp(name, "seg_min_len")) {
    if (value < (int64_t)PB_TILE) return fail(e, PBSIM_E_INVALID, "seg_min_len must be at least %u", PB_TILE);
    e->seg_min_len = value;
    return 0;
  }
  if (!strcmp(name, "pipeline")) {
    if (value < 0 || value > 2) return fail(e, PBSIM_E_INVALID, "pipeline must be 0, 1 or 2");
    if (e->running) return fail(e, PBSIM_E_INVALID, "pipeline cannot change during a run");
    e->pipeline = (int)value;
    return 0;
  }
  if (!strcmp(name, "sample_spec")) {
    e->sample_spec = value != 0;
    return 0;
  }
  if (!strcmp(name, "bam")) {
    if (e->running) return fail(e, PBSIM_E_INVALID, "bam cannot change during a run");
    e->bam = value != 0;
    return 0;
  }
  if (!strcmp(name, "align")) {
    if (e->running) return fail(e, PBSIM_E_INVALID, "align cannot change during a run");
    e->align = value != 0;
    return 0;
  }
  if (!strcmp(name, "deflate")) {
    if (e->running) return fail(e, PBSIM_E_INVALID, "deflate cannot change during a run");
    e->deflate = value != 0;
    return 0;
  }
  if (!strcmp(name, "first_batch_div")) {
    if (value < 1 || value > 64) return fail(e, PBSIM_E_INVALID, "first_batch_div must be 1..64");
    e->first_batch_div = value;
    return 0;
  }
  if (!strcmp(name, "host_batch_bases")) {
    if (value < 1) return fail(e, PBSIM_E_INVALID, "host_batch_bases must be positive");
    e->host_batch_bases = value;
    return 0;
  }
  if (!strcmp(name, "target_batch_bases")) {
    if (value < 1) return fail(e, PBSIM_E_INVALID, "target_batch_bases must be positive");
    e->target_batch_bases = value;
    return 0;
  }
  return fail(e, PBSIM_E_INVALID, "unknown option %s", name);
}

int pbsim_cuda_stats_device_block(pbsim_engine *e, void **dptr, int64_t *cells) {
  if (!e || !dptr || !cells || !e->model_set) return PBSIM_E_INVALID;
  *dptr = e->d_stats.p;
  *cells = e->stats_cells;
  return 0;
}

int pbsim_cuda_last_chunk_info(pbsim_engine *e, int64_t *out, int64_t cap_subreads, int64_t *n_subreads) {
  if (!e || !n_subreads) return PBSIM_E_INVALID;
  CK(cudaSetDevice(e->device));
  if (e->pipelined) return fail(e, PBSIM_E_INVALID, "last_chunk_info needs option pipeline = 0 (the producer has moved on)");
  const Batch &B = e->B;
  const uint32_t pass = (uint32_t)e->model.pass_num;
  const int64_t n = B.n_sub;
  *n_subreads = n;
  if (!out) return 0;
  const int64_t m = std::min<int64_t>(n, cap_subreads);
  std::vector<uint32_t> off(B.n_reads), wl(B.n_reads), meta(B.n_reads), rl(n), nc(n);
  CK(cudaMemcpy(off.data(), B.plan_off, (size_t)B.n_reads * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(wl.data(), B.plan_wlen, (size_t)B.n_reads * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(meta.data(), B.plan_meta, (size_t)B.n_reads * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(rl.data(), B.rlen, (size_t)n * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(nc.data(), B.ncol, (size_t)n * 4, cudaMemcpyDeviceToHost));
  for (int64_t s = 0; s < m; ++s) {
    const uint32_t r = (uint32_t)(s / pass);
    int64_t *o = out + s * 8;
    o[0] = (int64_t)B.first_read + 1 + r;
    o[1] = s % pass;
    o[2] = meta[r] & 0xFF;
    o[3] = off[r];
    o[4] = wl[r];
    o[5] = rl[s];
    o[6] = nc[s];
    o[7] = (meta[r] >> 8) & 1;
  }
  return 0;
}

}  // extern "C"
