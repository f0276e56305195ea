// pbsim (B200) — host driver: the reference's command line and file layout in front of libpbsim_cuda.
//
// Keeps the CLI surface of yukiteruono/pbsim3 (23 long options, pbsim.cpp:257-530), its defaults and
// validation (set_sim_param :1451-1688), the stderr report blocks (:5397-5465, :902-978, :5541-5564,
// :871-873) and the output layout <prefix>_NNNN.ref / .fq.gz / .maf.gz (:708-730, :939); the read
// generation itself is one simulate call per reference sequence into the CUDA engine (the seam of
// main :699-754).  Compression is in-process (zlib gzip members from a thread pool) instead of
// popen("gzip > file"); concatenated gzip members decompress to the same text.
//
// --strategy trans / templ (main :760-868) parse the transcript table / template FASTA here and hand the
// whole set to the engine (pbsim_cuda_set_seqset); outputs <prefix>.fq.gz / .maf.gz (:771-788).
//
// Engine-only options (additive): --gpu N, --rng philox|replay, --replay-draws F --replay-marks F,
// --threads N (host compression), --gzip gpu|host (default gpu: the records are gzip-compressed on the GPU and the
// driver only writes the members to the files; multi-pass output is <prefix>[_NNNN].bam, or SAM text in .sam.gz with
// --gzip host).  --method sample filters the FASTQ on the host (pbsim_host_sample_filter) and hands the pool to the engine.
#include <fcntl.h>
#include <getopt.h>
#include <sys/mman.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <deque>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pbsim_cuda.h"

namespace {

constexpr size_t kBufSize = 10240;          // BUF_SIZE
constexpr int kRefIdLenMax = 128;           // REF_ID_LEN_MAX
constexpr long kRefSeqNumMax = 9999;        // REF_SEQ_NUM_MAX
constexpr long kRefSeqLenMax = 1000000000;  // REF_SEQ_LEN_MAX
constexpr long kRefSeqLenMin = 100;         // REF_SEQ_LEN_MIN
constexpr int kFastqLenMax = 1000000;       // FASTQ_LEN_MAX
constexpr int kRatioMax = 1000;

struct Options {
  int set_flg[40] = {0};
  std::string strategy, method;
  std::string genome, transcript, templ, sample, profile_id, qshmm, errhmm;
  std::string prefix = "sd", id_prefix = "S";
  double depth = 20.0;
  long len_min = 100, len_max = 1000000;
  long sub_ratio = 6, ins_ratio = 55, del_ratio = 39;
  unsigned int seed = 0;
  double accuracy_min = 0.75, accuracy_max = 1.0, accuracy_mean = 0.85;
  double len_mean = 9000, len_sd = 7000;
  int pass_num = 1;
  double hp_del_bias = 1;
  // engine-only
  int gpu = 0;
  std::string rng = "philox", replay_draws, replay_marks;
  int threads = 0;
  int rank = 0, world = 1;   // one process per GPU: process `rank` of `world` simulates the sequences n with
                             // (n - 1) % world == rank (their output files are independent of everything else)
  std::string gzip = "gpu";  // who writes the gzip members: the GPU (gz_kernels.cuh) or zlib threads on the host
  std::string align = "maf"; // the second file: MAF blocks (.maf.gz) or SAM alignment lines (.aln.sam.gz)
};

std::thread *g_background = nullptr;  // a thread that must have ended before the process exits (CUDA start-up)

[[noreturn]] void die(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vfprintf(stderr, fmt, ap);
  va_end(ap);
  if (g_background && g_background->joinable() && g_background->get_id() != std::this_thread::get_id()) g_background->join();
  exit(-1);
}

long now_cpu() {
  struct rusage ru;
  getrusage(RUSAGE_SELF, &ru);
  return ru.ru_utime.tv_sec;
}
long now_wall() {
  struct timeval tv;
  gettimeofday(&tv, nullptr);
  return tv.tv_sec;
}

double now_seconds() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ------------------------------------------------------------------------------------------
// a few threads that copy byte ranges to file offsets: the gzip members the GPU wrote go from the engine's pinned
// staging buffers straight into the files, several 4 MiB blocks at a time.  The copies go through a shared mapping of
// the file (grown ahead with ftruncate, cut to its size at the end): write()/pwrite() on one file are serialised by
// the inode lock (3.5 GB/s measured on a RAM disk for the two output files together), page faults on a mapping are not.
// The reference's writers are the two `gzip > file` children (:708-730).
// ------------------------------------------------------------------------------------------
class WritePool {
 public:
  struct Range {
    int fd;
    const char *p;
    size_t n;
    uint64_t off;
  };
  explicit WritePool(int threads) {
    for (int i = 0; i < std::max(1, threads); ++i) workers_.emplace_back([this] { work(); });
  }
  ~WritePool() {
    {
      std::unique_lock<std::mutex> lk(mu_);
      closing_ = true;
      cv_work_.notify_all();
    }
    for (auto &t : workers_) t.join();
  }
  // returns when every byte is in the file (the caller's buffers are only valid until then); false on an I/O error.
  // The files must be large enough (GzipWriter::direct_range grows them).
  bool run(const std::vector<Range> &ranges) {
    constexpr size_t kBlock = 4 << 20;
    const size_t page = (size_t)sysconf(_SC_PAGESIZE);
    struct Map {
      char *base;
      size_t len;
    };
    std::vector<Map> maps;
    bool ok = true;
    {
      std::unique_lock<std::mutex> lk(mu_);
      for (const Range &r : ranges) {
        if (r.n == 0) continue;
        const uint64_t a = r.off / page * page;
        const size_t len = (size_t)(r.off + r.n - a);
        void *m = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_SHARED, r.fd, (off_t)a);
        if (m == MAP_FAILED) {  // a file that cannot be mapped (a pipe, some network file systems): plain pwrite
          for (size_t o = 0; o < r.n; o += kBlock) {
            queue_.push_back(Job{r.fd, nullptr, r.p + o, std::min(kBlock, r.n - o), r.off + o});
            ++open_;
          }
          continue;
        }
        maps.push_back(Map{static_cast<char *>(m), len});
        char *dst = static_cast<char *>(m) + (r.off - a);
        for (size_t o = 0; o < r.n; o += kBlock) {
          queue_.push_back(Job{-1, dst + o, r.p + o, std::min(kBlock, r.n - o), 0});
          ++open_;
        }
      }
      cv_work_.notify_all();
      cv_done_.wait(lk, [this] { return open_ == 0; });
      ok = !failed_;
    }
    for (const Map &m : maps) munmap(m.base, m.len);
    return ok;
  }

 private:
  struct Job {
    int fd;
    char *dst;
    const char *src;
    size_t n;
    uint64_t off;
  };
  void work() {
    for (;;) {
      Job j;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_work_.wait(lk, [this] { return closing_ || !queue_.empty(); });
        if (queue_.empty()) return;
        j = queue_.front();
        queue_.pop_front();
      }
      bool ok = true;
      if (j.dst) {
        memcpy(j.dst, j.src, j.n);
      } else {
        while (j.n > 0) {
          const ssize_t w = pwrite(j.fd, j.src, j.n, (off_t)j.off);
          if (w <= 0) {
            ok = false;
            break;
          }
          j.src += w;
          j.n -= (size_t)w;
          j.off += (uint64_t)w;
        }
      }
      std::unique_lock<std::mutex> lk(mu_);
      if (!ok) failed_ = true;
      if (--open_ == 0) cv_done_.notify_all();
    }
  }
  std::mutex mu_;
  std::condition_variable cv_work_, cv_done_;
  std::deque<Job> queue_;
  size_t open_ = 0;
  bool closing_ = false, failed_ = false;
  std::vector<std::thread> workers_;
};

// ------------------------------------------------------------------------------------------
// ordered gzip writer of one output file.  Text blocks (--gzip host, the SAM header) are compressed by zlib threads,
// one gzip member per block, and written in order; members that arrive compressed from the GPU bypass all of that
// (append_direct).  Every write is a pwrite at the file's running offset; an I/O or zlib error ends the run in close().
// ------------------------------------------------------------------------------------------
class GzipWriter {
 public:
  GzipWriter(const std::string &path, int threads, int level = 1) : path_(path), level_(level) {
    fd_ = open(path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd_ < 0) die("ERROR: Cannot open output file: %s\n", path.c_str());
    nthreads_ = std::max(1, threads);
  }
  // raw: the bytes are gzip members already: kept in order, not compressed
  void submit(const char *data, size_t n, bool raw = false) {
    if (n == 0) return;
    start_threads();
    std::unique_lock<std::mutex> lk(mu_);
    cv_space_.wait(lk, [this] { return pending_.size() + done_.size() < 64; });
    Job j;
    j.seq = next_seq_++;
    j.raw = raw;
    j.in.assign(data, data + n);
    pending_.push_back(std::move(j));
    cv_work_.notify_one();
  }
  // everything submitted so far is in the file
  void drain() {
    std::unique_lock<std::mutex> lk(mu_);
    cv_space_.wait(lk, [this] { return written_ == next_seq_; });
  }
  // the range WritePool::run needs to append n bytes behind what was submitted (drain() first)
  WritePool::Range direct_range(const char *p, size_t n) {
    WritePool::Range r{fd_, p, n, off_};
    off_ += n;
    bytes_out += n;
    // the pool copies through a mapping: the file has to be that long already (lengthened 1 GiB ahead; a file that
    // cannot be lengthened — a device, a pipe — is written with pwrite by the pool).  Measured on the GPU box's RAM disk
    // (profiles/r02_cli_wallclock.log): 16 threads copying into the two mapped files 4.3 GB/s, 16 pwrite threads 3.5
    // GB/s, allocating ahead with fallocate from a thread per file 3 GB/s — page allocation inside ONE file is
    // serialised by the file system (16 dd writers of 16 files: 45 GB/s), and the two output files are the layout
    if (off_ > size_) {
      size_ = (off_ + ((uint64_t)1 << 30)) & ~(((uint64_t)1 << 30) - 1);
      if (ftruncate(fd_, (off_t)size_) != 0) size_ = 0;
    }
    return r;
  }
  void fail() { failed_ = true; }
  void close() {
    {
      std::unique_lock<std::mutex> lk(mu_);
      closing_ = true;
      cv_work_.notify_all();
      cv_done_.notify_all();
    }
    for (auto &t : workers_) t.join();
    if (writer_.joinable()) writer_.join();
    if (size_ > off_ && ftruncate(fd_, (off_t)off_) != 0) failed_ = true;
    if (::close(fd_) != 0) failed_ = true;
    if (failed_) die("ERROR: Cannot write output file: %s\n", path_.c_str());
  }
  uint64_t bytes_in = 0, bytes_out = 0;

 private:
  struct Job {
    uint64_t seq;
    bool raw = false;
    std::vector<char> in, out;
  };
  void start_threads() {
    if (!workers_.empty()) return;
    for (int i = 0; i < nthreads_; ++i) workers_.emplace_back([this] { work(); });
    writer_ = std::thread([this] { write(); });
  }
  void work() {
    for (;;) {
      Job j;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_work_.wait(lk, [this] { return closing_ || !pending_.empty(); });
        if (pending_.empty()) return;
        j = std::move(pending_.front());
        pending_.pop_front();
      }
      bool ok = true;
      if (j.raw) {
        j.out.swap(j.in);
      } else {
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        ok = deflateInit2(&zs, level_, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) == Z_OK;
        if (ok) {
          j.out.resize(deflateBound(&zs, j.in.size()) + 64);
          zs.next_in = reinterpret_cast<Bytef *>(j.in.data());
          zs.avail_in = (uInt)j.in.size();
          zs.next_out = reinterpret_cast<Bytef *>(j.out.data());
          zs.avail_out = (uInt)j.out.size();
          ok = deflate(&zs, Z_FINISH) == Z_STREAM_END;
          j.out.resize(zs.total_out);
          deflateEnd(&zs);
        }
      }
      {
        std::unique_lock<std::mutex> lk(mu_);
        if (!ok) failed_ = true;
        bytes_in += j.raw ? j.out.size() : j.in.size();
        j.in.clear();
        j.in.shrink_to_fit();
        done_[j.seq] = std::move(j);
        cv_done_.notify_one();
      }
    }
  }
  void write() {
    uint64_t want = 0;
    for (;;) {
      Job j;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, [&] { return done_.count(want) || (closing_ && pending_.empty() && want == next_seq_); });
        if (!done_.count(want)) return;
        j = std::move(done_[want]);
        done_.erase(want);
        ++want;
      }
      const char *p = j.out.data();
      size_t n = j.out.size();
      bool ok = true;
      while (n > 0) {
        const ssize_t w = pwrite(fd_, p, n, (off_t)off_);
        if (w <= 0) {
          ok = false;
          break;
        }
        p += w;
        n -= (size_t)w;
        off_ += (uint64_t)w;
      }
      std::unique_lock<std::mutex> lk(mu_);
      if (!ok) failed_ = true;
      bytes_out += j.out.size();
      written_ = want;
      cv_space_.notify_all();
    }
  }
  std::string path_;
  int fd_ = -1;
  int level_, nthreads_ = 1;
  uint64_t size_ = 0;  // length the file was grown to for the mapped copies (cut back to off_ in close)
  uint64_t off_ = 0;  // the file's running offset: the writer thread's while jobs are pending, the caller's after drain()
  std::mutex mu_;
  std::condition_variable cv_work_, cv_done_, cv_space_;
  std::deque<Job> pending_;
  std::map<uint64_t, Job> done_;
  uint64_t next_seq_ = 0, written_ = 0;
  bool closing_ = false, failed_ = false;
  std::vector<std::thread> workers_;
  std::thread writer_;
};

// blocks for the compressor are cut at record-independent sizes; 8 MiB keeps members reasonably large
void stream_to(GzipWriter &w, const char *p, int64_t n, bool raw = false) {
  const int64_t blk = 8 << 20;
  for (int64_t o = 0; o < n; o += blk) w.submit(p + o, (size_t)std::min(blk, n - o), raw);
}

// one BGZF block (SAM spec 4.1) holding `data` (at most 64 KiB): the BAM file header goes through here, the
// alignment records arrive from the GPU as BGZF blocks already
std::string bgzf_block(const std::string &data) {
  z_stream zs;
  memset(&zs, 0, sizeof zs);
  deflateInit2(&zs, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
  std::string body(deflateBound(&zs, data.size()) + 16, '\0');
  zs.next_in = reinterpret_cast<Bytef *>(const_cast<char *>(data.data()));
  zs.avail_in = (uInt)data.size();
  zs.next_out = reinterpret_cast<Bytef *>(&body[0]);
  zs.avail_out = (uInt)body.size();
  deflate(&zs, Z_FINISH);
  body.resize(zs.total_out);
  deflateEnd(&zs);
  const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), reinterpret_cast<const Bytef *>(data.data()), (uInt)data.size());
  const uint32_t isize = (uint32_t)data.size();
  const uint16_t bsize = (uint16_t)(18 + body.size() + 8 - 1);
  std::string out;
  const unsigned char hdr[16] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0};
  out.append(reinterpret_cast<const char *>(hdr), 16);
  out.append(reinterpret_cast<const char *>(&bsize), 2);
  out += body;
  out.append(reinterpret_cast<const char *>(&crc), 4);
  out.append(reinterpret_cast<const char *>(&isize), 4);
  return out;
}

struct RefSeq {
  std::string id;
  long len = 0;
  std::string text;  // the sequence as get_genome_seq would re-read it from <prefix>_NNNN.ref; kept from the split
                     // pass so that every reference is read from disk once, not three times
};

// get_genome_inf (:896-991): split the multi-FASTA into <prefix>_NNNN.ref, collect lengths, print the block.
// The statement of the reference's fgets loop, line by line: the reader of files the parallel one declines.
std::vector<RefSeq> genome_inf_sequential(const Options &o) {
  fprintf(stderr, ":::: Reference stats ::::\n\n");
  fprintf(stderr, "file name : %s\n", o.genome.c_str());
  fprintf(stderr, "\n");
  FILE *fp = fopen(o.genome.c_str(), "r");
  if (!fp) die("ERROR: Cannot open file: %s\n", o.genome.c_str());
  setvbuf(fp, nullptr, _IOFBF, 8 << 20);
  std::vector<RefSeq> seqs;
  std::vector<char> line(kBufSize);
  FILE *out = nullptr;
  auto trim = [&](char *s) {
    size_t n = strlen(s);
    if (n && s[n - 1] == '\n') {
      s[n - 1] = '\0';
      return 1;
    }
    return 0;
  };
  auto finish = [&]() {
    if (seqs.back().len < kRefSeqLenMin) die("ERROR: Reference is too short. Acceptable length >= %ld.\n", kRefSeqLenMin);
    fprintf(stderr, "ref.%zu (len:%ld) : %s\n", seqs.size(), seqs.back().len, seqs.back().id.c_str());
    fclose(out);
  };
  while (fgets(line.data(), (int)kBufSize, fp)) {
    int ret = trim(line.data());
    if (line[0] == '>') {
      if (!seqs.empty()) finish();
      if ((long)seqs.size() + 1 > kRefSeqNumMax) die("ERROR: References are too many. Max number of reference is %ld.\n", kRefSeqNumMax);
      RefSeq r;
      r.id.assign(line.data() + 1, strnlen(line.data() + 1, kRefIdLenMax));
      seqs.push_back(r);
      char name[4096];
      snprintf(name, sizeof name, "%s_%04zu.ref", o.prefix.c_str(), seqs.size());
      out = fopen(o.rank == 0 ? name : "/dev/null", "w");  // one writer of the .ref files is enough
      if (!out) die("ERROR: Cannot open output file: %s\n", name);
      setvbuf(out, nullptr, _IOFBF, 8 << 20);
      while (ret != 1) {  // header longer than the buffer: skip its continuation
        if (!fgets(line.data(), (int)kBufSize, fp)) break;
        ret = trim(line.data());
      }
      fprintf(out, ">%s\n", seqs.back().id.c_str());
    } else {
      if (seqs.empty()) continue;  // text before the first header (the reference would crash here)
      const size_t ln = strlen(line.data());
      seqs.back().len += (long)ln;
      if (seqs.back().len > kRefSeqLenMax) die("ERROR: Reference is too long. Acceptable length <= %ld.\n", kRefSeqLenMax);
      fprintf(out, "%s\n", line.data());
      seqs.back().text.append(line.data(), ln);
    }
  }
  fclose(fp);
  if (seqs.empty()) die("ERROR: Reference is too short. Acceptable length >= %ld.\n", kRefSeqLenMin);
  finish();
  fprintf(stderr, "\n");
  return seqs;
}

// The same for ordinary FASTA files, in parallel (the 3.1 Gbp human genome is 44 million lines; the loop above spends
// 4-5 s on them).  The file is mapped; a first parallel scan finds the header lines ('>' at the start of a line), the
// longest line and any NUL byte; when every line fits one fgets buffer (so that the reference's chunking of long lines
// and its '>' test on chunk starts cannot matter) and no NUL cuts a line short, the records are independent: a thread
// per record collects its text and writes its .ref file (the body lines verbatim, which is what the fgets loop writes).
// Messages and errors are then replayed in the reference's order.  Returns false when the file is not of that kind.
bool genome_inf_parallel(const Options &o, int threads, std::vector<RefSeq> &seqs) {
  const int fd = open(o.genome.c_str(), O_RDONLY);
  if (fd < 0) return false;  // the sequential reader reports it
  struct stat sb;
  const char *min_env = getenv("PBSIM_INGEST_PARALLEL_MIN");  // tests: take this path for small files too
  const long min_bytes = min_env ? std::max(1L, atol(min_env)) : (1L << 16);  // small files: nothing to gain
  if (fstat(fd, &sb) != 0 || !S_ISREG(sb.st_mode) || sb.st_size < min_bytes) {
    close(fd);
    return false;
  }
  const size_t n = (size_t)sb.st_size;
  void *mp = mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (mp == MAP_FAILED) return false;
  madvise(mp, n, MADV_WILLNEED);
  const char *p = static_cast<const char *>(mp);
  const int T = std::max(1, std::min(threads, (int)(n >> 22) + 1));
  struct Slice {
    std::vector<size_t> headers;
    size_t first_nl = SIZE_MAX, last_nl = SIZE_MAX, max_gap = 0;
    bool nul = false;
  };
  std::vector<Slice> sl((size_t)T);
  {
    std::vector<std::thread> th;
    for (int t = 0; t < T; ++t)
      th.emplace_back([&, t] {
        const size_t a = n * (size_t)t / (size_t)T, b = n * (size_t)(t + 1) / (size_t)T;
        Slice &S = sl[(size_t)t];
        if (memchr(p + a, 0, b - a)) S.nul = true;
        size_t prev = SIZE_MAX;
        for (const char *q = p + a; q < p + b;) {
          const char *nl = static_cast<const char *>(memchr(q, '\n', (size_t)(p + b - q)));
          if (!nl) break;
          const size_t i = (size_t)(nl - p);
          if (prev == SIZE_MAX) S.first_nl = i;
          else S.max_gap = std::max(S.max_gap, i - prev - 1);
          prev = i;
          if (i + 1 < n && p[i + 1] == '>') S.headers.push_back(i + 1);
          q = nl + 1;
        }
        S.last_nl = prev;
      });
    for (auto &t : th) t.join();
  }
  std::vector<size_t> heads;
  if (p[0] == '>') heads.push_back(0);
  size_t longest = 0, prev = SIZE_MAX;  // prev: the newline in front of the current line (SIZE_MAX: start of file)
  bool nul = false;
  for (const Slice &S : sl) {
    nul |= S.nul;
    heads.insert(heads.end(), S.headers.begin(), S.headers.end());
    longest = std::max(longest, S.max_gap);
    if (S.first_nl != SIZE_MAX) {
      longest = std::max(longest, prev == SIZE_MAX ? S.first_nl : S.first_nl - prev - 1);
      prev = S.last_nl;
    }
  }
  longest = std::max(longest, prev == SIZE_MAX ? n : n - prev - 1);
  if (nul || longest > kBufSize - 2 || heads.empty()) {
    munmap(mp, n);
    return false;
  }
  const size_t R = std::min(heads.size(), (size_t)kRefSeqNumMax);  // the reader dies at header 10000 (below)
  seqs.assign(R, RefSeq());
  std::vector<int> open_failed(R, 0), write_failed(R, 0);
  std::atomic<size_t> next(0);
  auto parse = [&] {
    for (;;) {
      const size_t r = next.fetch_add(1);
      if (r >= R) return;
      const size_t a = heads[r], b = r + 1 < heads.size() ? heads[r + 1] : n;
      const char *hl = static_cast<const char *>(memchr(p + a, '\n', b - a));
      const size_t hend = hl ? (size_t)(hl - p) : b;  // end of the header line's text
      RefSeq &q = seqs[r];
      q.id.assign(p + a + 1, std::min(hend - a - 1, (size_t)kRefIdLenMax));
      const size_t body = hl ? hend + 1 : b;
      q.text.reserve(b - body);
      for (size_t i = body; i < b;) {
        const char *nl = static_cast<const char *>(memchr(p + i, '\n', b - i));
        const size_t e = nl ? (size_t)(nl - p) : b;
        q.text.append(p + i, e - i);
        i = e + 1;
      }
      q.len = (long)q.text.size();
      if (o.rank == 0) {  // one writer of the .ref files is enough
        char name[4096];
        snprintf(name, sizeof name, "%s_%04zu.ref", o.prefix.c_str(), r + 1);
        const int out = open(name, O_WRONLY | O_CREAT | O_TRUNC, 0644);
        if (out < 0) {
          open_failed[r] = 1;
          continue;
        }
        std::string head = ">" + q.id + "\n";
        bool ok = write(out, head.data(), head.size()) == (ssize_t)head.size();
        for (size_t i = body; ok && i < b;) {
          const ssize_t w = write(out, p + i, std::min(b - i, (size_t)1 << 30));
          if (w <= 0) ok = false;
          else i += (size_t)w;
        }
        if (ok && b > body && p[b - 1] != '\n') ok = write(out, "\n", 1) == 1;  // a last line without line feed
        if (close(out) != 0) ok = false;
        if (!ok) write_failed[r] = 1;
      }
    }
  };
  {
    std::vector<std::thread> th;
    for (int t = 0; t < std::max(1, std::min(threads, (int)R)); ++t) th.emplace_back(parse);
    for (auto &t : th) t.join();
  }
  munmap(mp, n);
  // the report and the checks, in the order the sequential loop makes them
  fprintf(stderr, ":::: Reference stats ::::\n\n");
  fprintf(stderr, "file name : %s\n", o.genome.c_str());
  fprintf(stderr, "\n");
  auto drop_later_refs = [&](size_t r) {  // the sequential reader has not come to the records behind r when it stops
    for (size_t q = r + 1; q < R && o.rank == 0; ++q) {
      char name[4096];
      snprintf(name, sizeof name, "%s_%04zu.ref", o.prefix.c_str(), q + 1);
      unlink(name);
    }
  };
  for (size_t r = 0; r < R; ++r) {
    if (open_failed[r] || write_failed[r] || seqs[r].len > kRefSeqLenMax || seqs[r].len < kRefSeqLenMin) drop_later_refs(r);
    if (open_failed[r]) die("ERROR: Cannot open output file: %s_%04zu.ref\n", o.prefix.c_str(), r + 1);
    if (write_failed[r]) die("ERROR: Cannot write output file: %s_%04zu.ref\n", o.prefix.c_str(), r + 1);
    if (seqs[r].len > kRefSeqLenMax) die("ERROR: Reference is too long. Acceptable length <= %ld.\n", kRefSeqLenMax);
    if (seqs[r].len < kRefSeqLenMin) die("ERROR: Reference is too short. Acceptable length >= %ld.\n", kRefSeqLenMin);
    fprintf(stderr, "ref.%zu (len:%ld) : %s\n", r + 1, seqs[r].len, seqs[r].id.c_str());
  }
  if (heads.size() > (size_t)kRefSeqNumMax) die("ERROR: References are too many. Max number of reference is %ld.\n", kRefSeqNumMax);
  fprintf(stderr, "\n");
  return true;
}

std::vector<RefSeq> genome_inf(const Options &o, int threads) {
  std::vector<RefSeq> seqs;
  if (genome_inf_parallel(o, threads, seqs)) return seqs;
  return genome_inf_sequential(o);
}

// ---- --strategy trans / templ: the sequence set the engine simulates in one run --------------------------------
struct SeqSetHost {
  std::vector<std::string> ids;
  std::vector<int32_t> plus, minus;
  std::string bases;
  std::vector<int64_t> start{0};
  long num = 0;             // transcript.num_seq / templ.num
  long total_exp = 0;       // transcript.total_exp
  long long len_total = 0;  // templ.len_total
};

int trim_line(char *s) {  // trim (:882-891)
  const size_t n = strlen(s);
  if (n && s[n - 1] == '\n') {
    s[n - 1] = '\0';
    return 1;
  }
  return 0;
}

// The transcript table as get_transcript_inf (:1075-1140) and the fgets loops of simulate_by_*_trans (:2748-2772)
// read it: one record per line, id <TAB> plus <TAB> minus <TAB> sequence, fields split the way strtok does (runs of
// tabs collapse); a line longer than the 10 KB buffer continues in the next fgets chunk, which is appended whole.
SeqSetHost read_transcripts(const Options &o) {
  FILE *fp = fopen(o.transcript.c_str(), "r");
  if (!fp) die("ERROR: Cannot open file: %s\n", o.transcript.c_str());
  SeqSetHost S;
  std::vector<char> line(kBufSize);
  int flg1 = 1;
  while (fgets(line.data(), (int)kBufSize, fp)) {
    const int flg2 = trim_line(line.data());
    if (flg1 == 1) {
      char *save = nullptr;
      const char *id = strtok_r(line.data(), "\t", &save);
      const char *pl = strtok_r(nullptr, "\t", &save);
      const char *mi = strtok_r(nullptr, "\t", &save);
      const char *sq = strtok_r(nullptr, "\t", &save);
      if (!id || !pl || !mi || !sq)
        die("ERROR: transcript record %ld does not have 4 tab-separated fields: %s\n", S.num + 1, o.transcript.c_str());
      S.num++;
      S.ids.emplace_back(id, strnlen(id, kRefIdLenMax));  // TRANS_ID_LEN_MAX = 128
      S.plus.push_back(atoi(pl));
      S.minus.push_back(atoi(mi));
      S.total_exp += S.plus.back() + S.minus.back();
      S.bases.append(sq);
    } else {
      S.bases.append(line.data());
    }
    if (flg2 == 1) S.start.push_back((int64_t)S.bases.size());
    flg1 = flg2;
  }
  fclose(fp);
  if (flg1 == 0 && !S.ids.empty()) {  // last record without a line feed: counted in the stats, never simulated (:2773)
    S.bases.resize((size_t)S.start.back());
    S.ids.pop_back();
    S.plus.pop_back();
    S.minus.pop_back();
  }
  fprintf(stderr, ":::: transcript stats ::::\n\n");  // print_transcript_stats (:1142-1149)
  fprintf(stderr, "file name : %s\n", o.transcript.c_str());
  fprintf(stderr, "transcript num : %ld\n", S.num);
  fprintf(stderr, "total expression value : %ld\n", S.total_exp);
  fprintf(stderr, "\n");
  return S;
}

// The template FASTA as get_templ_inf (:1366-1417) and simulate_by_*_templ (:3312-3329, :3560-3580) read it: header =
// text after '>' (128 characters kept), body lines concatenated; a template ends at the next header or at EOF and is
// simulated only if it holds at least one base.
SeqSetHost read_templates(const Options &o) {
  constexpr long kTemplateNumMax = 100000000, kTemplateLenMax = 1000000;  // :28-29
  FILE *fp = fopen(o.templ.c_str(), "r");
  if (!fp) die("ERROR: Cannot open file: %s\n", o.templ.c_str());
  SeqSetHost S;
  std::vector<char> line(kBufSize);
  std::string id, seq;
  bool have = false;
  auto flush = [&]() {
    if (have && !seq.empty()) {
      S.ids.push_back(id);
      S.plus.push_back(1);
      S.minus.push_back(0);
      S.bases.append(seq);
      S.start.push_back((int64_t)S.bases.size());
    }
    seq.clear();
  };
  while (fgets(line.data(), (int)kBufSize, fp)) {
    int ret = trim_line(line.data());
    if (line[0] == '>') {
      flush();
      S.num++;
      if (S.num > kTemplateNumMax) die("ERROR: template is too many. Max acceptable number is %ld.\n", kTemplateNumMax);
      id.assign(line.data() + 1, strnlen(line.data() + 1, kRefIdLenMax));
      have = true;
      while (ret != 1) {
        if (!fgets(line.data(), (int)kBufSize, fp)) break;
        ret = trim_line(line.data());
      }
    } else {
      const size_t n = strlen(line.data());
      seq.append(line.data(), n);
      S.len_total += (long long)n;
      if ((long)seq.size() > kTemplateLenMax) die("ERROR: template is too long. Max acceptable length is %ld.\n", kTemplateLenMax);
      have = true;  // text before the first header is a template with the (empty) id the reference starts with
    }
  }
  flush();
  fclose(fp);
  fprintf(stderr, ":::: Template stats ::::\n\n");  // print_templ_stats (:1424-1431)
  fprintf(stderr, "file name : %s\n", o.templ.c_str());
  fprintf(stderr, "template num. : %ld\n", S.num);
  fprintf(stderr, "template total length : %lld\n", S.len_total);
  fprintf(stderr, "\n");
  return S;
}

void print_help() {
  fprintf(stderr,
          "\nUSAGE: pbsim [options] \n\n [general options]\n\n"
          "  --prefix             prefix of output files (sd).\n"
          "  --id-prefix          prefix of read ID (S).\n"
          "  --seed               for a pseudorandom number generator (Unix time).\n\n"
          " [options for whole genome sequencing]\n\n"
          "  --strategy           wgs\n"
          "  --genome             FASTA format file (text file only).\n"
          "  --depth              depth of coverage (20.0).\n"
          "  --length-min         minimum length (100).\n"
          "  --length-max         maximum length (1000000).\n\n"
          " [options for quality score model]\n\n"
          "  --method             qshmm\n"
          "  --qshmm              quality score model.\n"
          "  --length-mean        mean length (9000.0).\n"
          "  --length-sd          standard deviation of length (7000.0).\n"
          "  --accuracy-mean      mean accuracy (0.85).\n"
          "  --pass-num           number of sequencing passes (1).\n"
          "  --difference-ratio   difference (error) ratio (6:55:39).\n"
          "  --hp-del-bias        bias intensity of deletion in homopolymer (1).\n\n"
          " [options for error model]\n\n"
          "  --method             errhmm\n"
          "  --errhmm             error model.\n\n"
          " [B200 engine]\n\n"
          "  --gpu                CUDA device ordinal (0).\n"
          "  --rng                philox (default) | replay\n"
          "  --replay-draws       int32 log of the reference's rand() draws (replay mode).\n"
          "  --replay-marks       int64 draw count after every (read, pass) (replay mode).\n"
          "  --threads            compression threads (hardware concurrency).\n"
          "  --rank R --world N   one process per GPU: this process simulates the sequences n with (n-1) %% N == R\n"
          "                       (WGS; every process reads the whole genome, files are written per sequence).\n"
          "  --gzip               gpu (default): gzip members / BGZF blocks are written on the GPU (multi-pass\n"
          "                       output is <prefix>_NNNN.bam) | host: zlib threads (multi-pass: .sam.gz).\n"
          "  --align              maf (default): alignments as MAF, <prefix>_NNNN.maf.gz | sam: each read's true\n"
          "                       alignment as a SAM line with a CIGAR, <prefix>_NNNN.aln.sam.gz (with --pass-num > 1\n"
          "                       it needs --gzip host).\n\n"
          " [options for transcriptome / template sequencing]\n\n"
          "  --strategy           trans | templ\n"
          "  --transcript         transcript table: id, plus count, minus count, sequence (tab separated).\n"
          "  --template           FASTA file of templates; every template is read once, in full.\n\n"
          " [options for sampling-based simulation]\n\n"
          "  --method             sample\n"
          "  --sample             FASTQ format file to sample.\n"
          "  --sample-profile-id  sample (filtered) profile ID; with --sample the profile is stored, without it reused.\n"
          "  --accuracy-min       minimum accuracy (0.75).\n"
          "  --accuracy-max       maximum accuracy (1.00).\n\n");
}

template <class T>
std::vector<T> read_binary(const std::string &path) {
  FILE *fp = fopen(path.c_str(), "rb");
  if (!fp) die("ERROR: Cannot open file: %s\n", path.c_str());
  fseek(fp, 0, SEEK_END);
  long n = ftell(fp);
  fseek(fp, 0, SEEK_SET);
  std::vector<T> v((size_t)n / sizeof(T));
  if (!v.empty() && fread(v.data(), sizeof(T), v.size(), fp) != v.size()) die("ERROR: short read: %s\n", path.c_str());
  fclose(fp);
  return v;
}

}  // namespace

int main(int argc, char **argv) {
  const long rst1 = now_cpu(), t1 = now_wall();
  Options o;
  o.seed = (unsigned int)time(nullptr);
  static struct option long_options[] = {
      {"strategy", 1, nullptr, 0},   {"method", 1, nullptr, 0},         {"genome", 1, nullptr, 0},
      {"transcript", 1, nullptr, 0}, {"prefix", 1, nullptr, 0},         {"id-prefix", 1, nullptr, 0},
      {"depth", 1, nullptr, 0},      {"length-min", 1, nullptr, 0},     {"length-max", 1, nullptr, 0},
      {"difference-ratio", 1, nullptr, 0}, {"seed", 1, nullptr, 0},     {"sample", 1, nullptr, 0},
      {"sample-profile-id", 1, nullptr, 0}, {"accuracy-min", 1, nullptr, 0}, {"accuracy-max", 1, nullptr, 0},
      {"qshmm", 1, nullptr, 0},      {"errhmm", 1, nullptr, 0},         {"length-mean", 1, nullptr, 0},
      {"length-sd", 1, nullptr, 0},  {"accuracy-mean", 1, nullptr, 0},  {"pass-num", 1, nullptr, 0},
      {"template", 1, nullptr, 0},   {"hp-del-bias", 1, nullptr, 0},
      // engine-only
      {"gpu", 1, nullptr, 0},        {"rng", 1, nullptr, 0},            {"replay-draws", 1, nullptr, 0},
      {"replay-marks", 1, nullptr, 0}, {"threads", 1, nullptr, 0},      {"gzip", 1, nullptr, 0},
      {"rank", 1, nullptr, 0},       {"world", 1, nullptr, 0},          {"align", 1, nullptr, 0},
      {nullptr, 0, nullptr, 0}};
  int opt, idx = 0;
  while ((opt = getopt_long(argc, argv, "", long_options, &idx)) != -1) {
    if (opt != 0) exit(-1);
    o.set_flg[idx] = 1;
    const char *a = optarg;
    switch (idx) {
      case 0:
        if (!strncmp(a, "wgs", 3)) o.strategy = "wgs";
        else if (!strncmp(a, "trans", 5)) o.strategy = "trans";
        else if (!strncmp(a, "templ", 5)) o.strategy = "templ";
        else die("ERROR (strategy: %s): Acceptable value: wgs, trans, templ.\n", a);
        break;
      case 1:
        if (!strncmp(a, "qshmm", 5)) o.method = "qshmm";
        else if (!strncmp(a, "errhmm", 6)) o.method = "errhmm";
        else if (!strncmp(a, "sample", 6)) o.method = "sample";
        else die("ERROR (method: %s): Acceptable value: qshmm, errhmm, sample.\n", a);
        break;
      case 2: o.genome = a; break;
      case 3: o.transcript = a; break;
      case 4: o.prefix = a; break;
      case 5: o.id_prefix = a; break;
      case 6:
        o.depth = atof(a);
        if (o.depth <= 0.0) die("ERROR (depth: %s): Acceptable range is more than 0.\n", a);
        break;
      case 7:
        if (strlen(a) >= 8) die("ERROR (length-min: %s): Acceptable range is 1-%d.\n", a, kFastqLenMax);
        o.len_min = atoi(a);
        if (o.len_min < 1 || o.len_min > kFastqLenMax) die("ERROR (length-min: %s): Acceptable range is 1-%d.\n", a, kFastqLenMax);
        break;
      case 8:
        if (strlen(a) >= 8) die("ERROR (length-max: %s): Acceptable range is 1-%d.\n", a, kFastqLenMax);
        o.len_max = atoi(a);
        if (o.len_max < 1 || o.len_max > kFastqLenMax) die("ERROR (length-max: %s): Acceptable range is 1-%d.\n", a, kFastqLenMax);
        break;
      case 9: {
        std::string tmp(a);
        char *save = nullptr;
        char *tp = strtok_r(&tmp[0], ":", &save);
        for (int num = 0; num < 3; ++num) {
          if (!tp) die("ERROR (difference-ratio: %s): Format is sub:ins:del.\n", a);
          if (strlen(tp) >= 5) die("ERROR (difference-ratio: %s): Acceptable range is 0-%d.\n", a, kRatioMax);
          long r = atoi(tp);
          if (r < 0 || r > kRatioMax) die("ERROR (difference-ratio: %s): Acceptable range is 0-%d.\n", a, kRatioMax);
          (num == 0 ? o.sub_ratio : num == 1 ? o.ins_ratio : o.del_ratio) = r;
          tp = strtok_r(nullptr, ":", &save);
        }
        break;
      }
      case 10: o.seed = (unsigned int)atoi(a); break;
      case 11: o.sample = a; break;
      case 12: o.profile_id = a; break;
      case 13:
        o.accuracy_min = atof(a);
        if (o.accuracy_min < 0.0 || o.accuracy_min > 1.0) die("ERROR (accuracy-min: %s): Acceptable range is 0.0-1.0.\n", a);
        break;
      case 14:
        o.accuracy_max = atof(a);
        if (o.accuracy_max < 0.0 || o.accuracy_max > 1.0) die("ERROR (accuracy-max: %s): Acceptable range is 0.0-1.0.\n", a);
        break;
      case 15: o.qshmm = a; break;
      case 16: o.errhmm = a; break;
      case 17:
        o.len_mean = atof(a);
        if (o.len_mean < 1 || o.len_mean > kFastqLenMax) die("ERROR (length-mean: %s): Acceptable range is 1-%d.\n", a, kFastqLenMax);
        break;
      case 18:
        o.len_sd = atof(a);
        if (o.len_sd < 0 || o.len_sd > kFastqLenMax) die("ERROR (length-sd: %s): Acceptable range is 0-%d.\n", a, kFastqLenMax);
        break;
      case 19:
        o.accuracy_mean = atof(a);
        if (o.accuracy_mean < 0.0 || o.accuracy_mean > 1.0) die("ERROR (accuracy-mean: %s): Acceptable range is 0.0-1.0.\n", a);
        break;
      case 20:
        o.pass_num = atoi(a);
        if (o.pass_num < 1) die("ERROR (pass_num: %s): Acceptable range is more than 1.\n", a);
        break;
      case 21: o.templ = a; break;
      case 22:
        if (strlen(a) >= 8) die("ERROR (hp-del-bias: %s): Acceptable range is 1-10.\n", a);
        o.hp_del_bias = atof(a);
        if (o.hp_del_bias < 1 || o.hp_del_bias > 10) die("ERROR (hp-del-bias: %s): Acceptable range is 1-10.\n", a);
        break;
      case 23: o.gpu = atoi(a); break;
      case 24: o.rng = a; break;
      case 25: o.replay_draws = a; break;
      case 26: o.replay_marks = a; break;
      case 27: o.threads = atoi(a); break;
      case 29: o.rank = atoi(a); break;
      case 30: o.world = atoi(a); break;
      case 28:
        if (!strcmp(a, "gpu") || !strcmp(a, "host")) o.gzip = a;
        else die("ERROR (gzip: %s): Acceptable value: gpu, host.\n", a);
        break;
      case 31:
        if (!strcmp(a, "maf") || !strcmp(a, "sam")) o.align = a;
        else die("ERROR (align: %s): Acceptable value: maf, sam.\n", a);
        break;
      default: break;
    }
  }
  if (argc == 1) {
    print_help();
    exit(-1);
  }
  // ---- set_sim_param (:1451-1688)
  if (!o.set_flg[0] || !o.set_flg[1]) die("ERROR: --strategy and --method must be set.\n");
  if (o.strategy != "wgs" && o.method == "sample") die("ERROR: sampling-based simulation is possible only for wgs strategy.\n");
  if (o.strategy == "wgs" && !o.set_flg[2]) die("ERROR: for --strategy wgs, --genome must be set.\n");
  if (o.strategy == "trans" && !o.set_flg[3]) die("ERROR: for --strategy trans, --transcript must be set.\n");
  if (o.strategy == "templ" && !o.set_flg[21]) die("ERROR: for --strategy templ, --template must be set.\n");
  if (o.method == "qshmm" && !o.set_flg[15]) die("ERROR: for --method qshmm, --qshmm must be set.\n");
  if (o.method == "errhmm" && !o.set_flg[16]) die("ERROR: for --method errhmm, --errhmm must be set.\n");
  // sample, sample-profile-id (:1565-1616): --sample alone filters the FASTQ, with a profile id the filtered reads are
  // stored (sample_profile_<id>.fastq / .stats), the id alone reuses a stored profile
  const bool sample = o.method == "sample";
  int sample_mode = 0;  // 0: METHOD_SAM, 1: METHOD_SAM_STORE, 2: METHOD_SAM_REUSE
  std::string profile_fq, profile_stats;
  if (sample) {
    if (o.set_flg[11]) sample_mode = o.set_flg[12] ? 1 : 0;
    else if (o.set_flg[12]) sample_mode = 2;
    else die("ERROR: for --method sample, --sample (and/or --sample-profile-id) must be set.\n");
  }
  if (o.set_flg[12]) {
    profile_fq = "sample_profile_" + o.profile_id + ".fastq";
    profile_stats = "sample_profile_" + o.profile_id + ".stats";
  }
  auto readable = [](const std::string &f) {
    FILE *fp = fopen(f.c_str(), "r");
    if (fp) fclose(fp);
    return fp != nullptr;
  };
  if (sample_mode == 1) {
    if (readable(profile_fq)) die("ERROR: %s exists.\n", profile_fq.c_str());
    if (readable(profile_stats)) die("ERROR: %s exists.\n", profile_stats.c_str());
  }
  if (sample_mode == 2) {
    if (!readable(profile_fq)) die("ERROR: %s does not exist.\n", profile_fq.c_str());
    if (!readable(profile_stats)) die("ERROR: %s does not exist.\n", profile_stats.c_str());
  }
  if (o.set_flg[13]) o.accuracy_min = int(o.accuracy_min * 100) * 0.01;
  if (o.set_flg[14]) o.accuracy_max = int(o.accuracy_max * 100) * 0.01;
  if (o.set_flg[19]) o.accuracy_mean = int(o.accuracy_mean * 100) * 0.01;
  if (o.len_min > o.len_max) die("ERROR: length min(%ld) is greater than max(%ld).\n", o.len_min, o.len_max);
  if (o.world < 1 || o.rank < 0 || o.rank >= o.world) die("ERROR: --rank must be in 0..world-1.\n");
  if (o.world > 1 && (o.strategy != "wgs" || o.rng == "replay"))
    die("ERROR: --world > 1 shards the sequences of --strategy wgs in philox mode; shard a transcript table by read range through the library instead.\n");
  if (o.pass_num > 1 && sample) die("ERROR: sampling-based simulation supports only single-pass.\n");  // :1675-1679
  const bool qs = o.method == "qshmm";
  const bool wgs = o.strategy == "wgs";

  // ---- print_sim_param (:5397-5465)
  fprintf(stderr, ":::: Simulation parameters :::\n\n");
  fprintf(stderr, "strategy : %s\n", o.strategy.c_str());
  fprintf(stderr, "method : %s\n", o.method.c_str());
  if (!sample) fprintf(stderr, "%s : %s\n", o.method.c_str(), qs ? o.qshmm.c_str() : o.errhmm.c_str());
  if (wgs) fprintf(stderr, "genome : %s\n", o.genome.c_str());
  else if (o.strategy == "trans") fprintf(stderr, "transcript : %s\n", o.transcript.c_str());
  else fprintf(stderr, "template : %s\n", o.templ.c_str());
  fprintf(stderr, "prefix : %s\n", o.prefix.c_str());
  fprintf(stderr, "id-prefix : %s\n", o.id_prefix.c_str());
  if (wgs) fprintf(stderr, "depth : %lf\n", o.depth);
  if (sample) {
    fprintf(stderr, "length-mean : (sample FASTQ)\n");
    fprintf(stderr, "length-sd : (sample FASTQ)\n");
    fprintf(stderr, "length-min : %ld\n", o.len_min);
    fprintf(stderr, "length-max : %ld\n", o.len_max);
  } else if (o.strategy != "templ") {
    fprintf(stderr, "length-mean : %f\n", o.len_mean);
    fprintf(stderr, "length-sd : %f\n", o.len_sd);
    fprintf(stderr, "length-min : %ld\n", o.len_min);
    fprintf(stderr, "length-max : %ld\n", o.len_max);
  }
  if (qs || sample) fprintf(stderr, "difference-ratio : %ld:%ld:%ld\n", o.sub_ratio, o.ins_ratio, o.del_ratio);
  fprintf(stderr, "seed : %d\n", o.seed);
  if (sample) {  // printf("%s", NULL) prints "(null)" with glibc
    fprintf(stderr, "sample : %s\n", o.set_flg[11] ? o.sample.c_str() : "(null)");
    fprintf(stderr, "sample-profile-id : %s\n", o.set_flg[12] ? o.profile_id.c_str() : "(null)");
    fprintf(stderr, "accuracy-mean : (sample FASTQ)\n");
    fprintf(stderr, "accuracy-sd : (sample FASTQ)\n");
    fprintf(stderr, "accuracy-min : %f\n", o.accuracy_min);
    fprintf(stderr, "accuracy-max : %f\n", o.accuracy_max);
  } else {
    fprintf(stderr, "accuracy-mean : %f\n", o.accuracy_mean);
  }
  fprintf(stderr, "pass_num : %d\n", o.pass_num);
  fprintf(stderr, "hp-del-bias : %f\n", o.hp_del_bias);
  fprintf(stderr, "\n");

  // ---- sample reads (main :579-616): get_sample_inf + print_sample_stats
  std::string pool_q;
  std::vector<int64_t> pool_start{0};
  if (sample) {
    pbsim_sample_stats ss;
    memset(&ss, 0, sizeof ss);
    auto slurp = [](const std::string &f, std::string *out) {
      FILE *fp = fopen(f.c_str(), "rb");
      if (!fp) return false;
      char buf[1 << 16];
      size_t k;
      while ((k = fread(buf, 1, sizeof buf, fp)) > 0) out->append(buf, k);
      fclose(fp);
      return true;
    };
    if (sample_mode == 2) {
      // the stored profile: statistics as the reference wrote them (:1317-1326), one quality string per line
      std::string text, line;
      if (!slurp(profile_stats, &text) || !slurp(profile_fq, &pool_q)) die("ERROR: Cannot open sample_profile\n");
      size_t p = 0;
      while (p < text.size()) {
        size_t q = text.find('\n', p);
        if (q == std::string::npos) q = text.size();
        line = text.substr(p, q - p);
        p = q + 1;
        const size_t tab = line.find('\t');
        if (tab == std::string::npos) continue;
        const std::string item = line.substr(0, tab), val = line.substr(tab + 1);
        if (item == "num") ss.num_filtered = atol(val.c_str());
        else if (item == "len_total") ss.len_total_filtered = atol(val.c_str());
        else if (item == "len_min") ss.len_min_filtered = atol(val.c_str());
        else if (item == "len_max") ss.len_max_filtered = atol(val.c_str());
        else if (item == "len_mean") ss.len_mean_filtered = atof(val.c_str());
        else if (item == "len_sd") ss.len_sd_filtered = atof(val.c_str());
        else if (item == "accuracy_mean") ss.accuracy_mean_filtered = atof(val.c_str());
        else if (item == "accuracy_sd") ss.accuracy_sd_filtered = atof(val.c_str());
      }
      std::string packed;
      for (size_t a = 0; a < pool_q.size();) {
        size_t b = pool_q.find('\n', a);
        if (b == std::string::npos) b = pool_q.size();
        packed.append(pool_q, a, b - a);
        pool_start.push_back((int64_t)packed.size());
        a = b + 1;
      }
      pool_q.swap(packed);
      if ((int64_t)pool_start.size() - 1 != ss.num_filtered || (int64_t)pool_q.size() != ss.len_total_filtered)
        die("ERROR: %s does not match %s.\n", profile_fq.c_str(), profile_stats.c_str());
    } else {
      std::string fq;
      if (!slurp(o.sample, &fq)) die("ERROR: Cannot open file: %s\n", o.sample.c_str());
      pool_q.resize(fq.size() + 1);
      pool_start.assign((size_t)std::count(fq.begin(), fq.end(), '\n') / 4 + 2, 0);
      int64_t n = 0;
      const char *ferr = nullptr;
      if (pbsim_host_sample_filter(fq.data(), (int64_t)fq.size(), o.len_min, o.len_max, o.accuracy_min, o.accuracy_max,
                                   &pool_q[0], pool_start.data(), (int64_t)pool_start.size(), &n, &ss, &ferr) != 0)
        die("%s\n", ferr);
      pool_start.resize((size_t)n + 1);
      pool_q.resize((size_t)pool_start[n]);
      if (sample_mode == 1) {
        FILE *f1 = fopen(profile_fq.c_str(), "w"), *f2 = fopen(profile_stats.c_str(), "w");
        if (!f1 || !f2) die("ERROR: Cannot open sample_profile\n");
        for (int64_t i = 0; i < n; ++i) {
          fwrite(pool_q.data() + pool_start[i], 1, (size_t)(pool_start[i + 1] - pool_start[i]), f1);
          fputc('\n', f1);
        }
        fprintf(f2, "num\t%ld\n", (long)ss.num_filtered);
        fprintf(f2, "len_total\t%lld\n", (long long)ss.len_total_filtered);
        fprintf(f2, "len_min\t%ld\n", (long)ss.len_min_filtered);
        fprintf(f2, "len_max\t%ld\n", (long)ss.len_max_filtered);
        fprintf(f2, "len_mean\t%f\n", ss.len_mean_filtered);
        fprintf(f2, "len_sd\t%f\n", ss.len_sd_filtered);
        fprintf(f2, "accuracy_mean\t%f\n", ss.accuracy_mean_filtered);
        fprintf(f2, "accuracy_sd\t%f\n", ss.accuracy_sd_filtered);
        fclose(f1);
        fclose(f2);
      }
    }
    // print_sample_stats (:1336-1358)
    fprintf(stderr, ":::: sample reads stats ::::\n\n");
    if (sample_mode == 2) {
      fprintf(stderr, "file name : %s\n", profile_fq.c_str());
    } else {
      fprintf(stderr, "file name : %s\n", o.sample.c_str());
      fprintf(stderr, "\n:: all reads ::\n");
      fprintf(stderr, "read num. : %ld\n", (long)ss.num);
      fprintf(stderr, "read total length : %lld\n", (long long)ss.len_total);
      fprintf(stderr, "read min length : %ld\n", (long)ss.len_min);
      fprintf(stderr, "read max length : %ld\n", (long)ss.len_max);
    }
    fprintf(stderr, "\n:: filtered reads ::\n");
    fprintf(stderr, "read num. : %ld\n", (long)ss.num_filtered);
    fprintf(stderr, "read total length : %lld\n", (long long)ss.len_total_filtered);
    fprintf(stderr, "read min length : %ld\n", (long)ss.len_min_filtered);
    fprintf(stderr, "read max length : %ld\n", (long)ss.len_max_filtered);
    fprintf(stderr, "read length mean (SD) : %f (%f)\n", ss.len_mean_filtered, ss.len_sd_filtered);
    fprintf(stderr, "read accuracy mean (SD) : %f (%f)\n", ss.accuracy_mean_filtered, ss.accuracy_sd_filtered);
    fprintf(stderr, "\n");
  }

  // ---- model + tables (set_qshmm/set_errhmm/set_mut + table builders)
  pbsim_host_params hp;
  memset(&hp, 0, sizeof hp);
  hp.method = sample ? PBSIM_METHOD_SAMPLE : (qs ? PBSIM_METHOD_QSHMM : PBSIM_METHOD_ERRHMM);
  hp.pass_num = o.pass_num;
  hp.len_min = o.len_min;
  hp.len_max = o.len_max;
  hp.len_mean = o.len_mean;
  hp.len_sd = o.len_sd;
  hp.accuracy_mean = o.accuracy_mean;
  hp.sub_ratio = o.sub_ratio;
  hp.ins_ratio = o.ins_ratio;
  hp.del_ratio = o.del_ratio;
  snprintf(hp.id_prefix, sizeof hp.id_prefix, "%s", o.id_prefix.c_str());
  pbsim_host_model *hm = nullptr;
  const char *err = nullptr;
  const std::string model_path = qs ? o.qshmm : o.errhmm;
  if (pbsim_host_model_load(&hm, &hp, sample ? nullptr : model_path.c_str(), &err) != 0) {
    if (strstr(err, "Cannot open")) die("ERROR: Cannot open file: %s\n", model_path.c_str());
    die("%s\n", err);
  }
  // ---- the input files are read before the GPU is touched, in the reference's order (get_genome_inf :896 /
  //      get_transcript_inf :1075 / get_templ_inf :1366 come right after the model): their errors and stats blocks
  //      appear exactly where the reference prints them
  const bool trans = o.strategy == "trans";
  std::vector<RefSeq> seqs;
  SeqSetHost S;
  // (the CUDA context comes up on a thread of its own meanwhile; its outcome is looked at afterwards)
  const int threads = o.threads > 0 ? o.threads : std::max(2u, std::thread::hardware_concurrency());
  pbsim_engine *eng = nullptr;
  int create_rc = 0;
  std::string create_err;
  std::thread creator([&] {
    create_rc = pbsim_cuda_create(&eng, o.gpu);
    if (create_rc != 0) create_err = pbsim_cuda_last_error(nullptr);  // thread-local in the library: read it here
  });
  g_background = &creator;
  const double t_load0 = now_seconds();
  if (wgs) seqs = genome_inf(o, threads);
  else S = trans ? read_transcripts(o) : read_templates(o);
  const double load_seconds = now_seconds() - t_load0;
  creator.join();
  g_background = nullptr;
  if (create_rc != 0) die("ERROR: %s\n", create_err.c_str());
  if (pbsim_cuda_set_model(eng, pbsim_host_model_get(hm)) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
  if (pbsim_cuda_set_option(eng, "deflate", o.gzip == "gpu" ? 1 : 0) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
  if (sample && pbsim_cuda_set_pool(eng, pool_q.data(), pool_start.data(), (int64_t)pool_start.size() - 1) != 0)
    die("ERROR: %s\n", pbsim_cuda_last_error(eng));

  // ---- replay inputs
  std::vector<int32_t> draws;
  std::vector<int64_t> marks, starts;
  const bool replay = o.rng == "replay";
  if (replay) {
    draws = read_binary<int32_t>(o.replay_draws);
    marks = read_binary<int64_t>(o.replay_marks);
    starts.resize(marks.size());
    for (size_t i = 0; i < marks.size(); ++i) starts[i] = i == 0 ? 0 : marks[i - 1];
  }
  size_t replay_pos = 0;
  WritePool pool(std::min(threads, 16));
  double gen_seconds = 0, write_seconds = 0, chunk_wait_seconds = 0;
  int64_t written_bytes = 0;
  int64_t total_bases = 0;
  double bias[12] = {0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0};

  // one simulate call of the reference: stream the engine's chunks into the two compressed files
  // multi-pass output: <stem>.bam like the reference (:715-722) when the GPU writes the BGZF blocks, SAM text in
  // <stem>.sam.gz with --gzip host
  const bool bam = o.pass_num > 1 && o.gzip == "gpu";
  if (pbsim_cuda_set_option(eng, "bam", bam ? 1 : 0) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
  const bool align = o.align == "sam";
  if (align && bam) die("ERROR: --align sam with --pass-num > 1 needs --gzip host (BAM reads and SAM alignment lines are not written together).\n");
  if (pbsim_cuda_set_option(eng, "align", align ? 1 : 0) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
  // sq: the @SQ lines of the alignment file (--align sam)
  auto simulate_to_files = [&](const std::string &stem, const std::string &pu, int64_t len_quota, const std::string &sq) {
    GzipWriter reads_out((stem + (o.pass_num == 1 ? ".fq.gz" : (bam ? ".bam" : ".sam.gz"))).c_str(), std::max(1, threads / 2));
    GzipWriter maf_out((stem + (align ? ".aln.sam.gz" : ".maf.gz")).c_str(), std::max(1, threads / 2));
    if (align) {
      const std::string h = "@HD\tVN:1.6\tSO:unknown\n" + sq + "@PG\tID:pbsim\tPN:pbsim\n";
      maf_out.submit(h.data(), h.size());
    }
    if (o.pass_num > 1) {  // SAM header (:721-722, :781-782)
      char hdr[1024];
      int m = snprintf(hdr, sizeof hdr,
                       "@HD\tVN:1.5\tSO:unknown\tpb:3.0.7\n@RG\tID:ffffffff\tPL:PACBIO\tDS:READTYPE=SUBREAD;Ipd:CodecV1=ip;"
                       "PulseWidth:CodecV1=pw;BINDINGKIT=101-789-500;SEQUENCINGKIT=101-826-100;BASECALLERVERSION=5.0.0;"
                       "FRAMERATEHZ=100.000000\tPU:%s\tPM:SEQUELII\n",
                       pu.c_str());
      if (bam) {
        // BAM file header (SAM spec 4.2): magic, the header text, no reference sequences — as one BGZF block
        std::string h("BAM\1", 4);
        const uint32_t l_text = (uint32_t)m, n_ref = 0;
        h.append(reinterpret_cast<const char *>(&l_text), 4);
        h.append(hdr, (size_t)m);
        h.append(reinterpret_cast<const char *>(&n_ref), 4);
        const std::string blk = bgzf_block(h);
        reads_out.submit(blk.data(), blk.size(), true);
      } else {
        reads_out.submit(hdr, (size_t)m);
      }
    }
    pbsim_run run;
    memset(&run, 0, sizeof run);
    run.rng_mode = replay ? PBSIM_RNG_REPLAY : PBSIM_RNG_PHILOX;
    run.seed = o.seed;
    run.len_quota = len_quota;
    if (replay) {
      run.replay_draws = draws.data();
      run.replay_ndraws = (int64_t)draws.size();
      run.replay_starts = starts.data() + replay_pos;
      run.replay_nsubreads = (int64_t)(starts.size() - replay_pos);
    }
    if (pbsim_cuda_simulate_begin(eng, &run) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    for (;;) {
      pbsim_chunk c;
      const double tc = now_seconds();
      const int rc = pbsim_cuda_next_chunk(eng, &c);
      chunk_wait_seconds += now_seconds() - tc;
      if (rc < 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
      if (rc == 0) break;
      if (c.compressed) {
        // gzip members / BGZF blocks written by the GPU: from the engine's pinned staging straight into the files
        reads_out.drain();
        maf_out.drain();
        std::vector<WritePool::Range> ranges;
        if (c.reads_bytes) ranges.push_back(reads_out.direct_range(c.reads, (size_t)c.reads_bytes));
        if (c.maf_bytes) ranges.push_back(maf_out.direct_range(c.maf, (size_t)c.maf_bytes));
        const double tw = now_seconds();
        if (!pool.run(ranges)) {
          reads_out.fail();
          maf_out.fail();
        }
        write_seconds += now_seconds() - tw;
        written_bytes += c.reads_bytes + c.maf_bytes;
      } else {
        stream_to(reads_out, c.reads, c.reads_bytes);
        stream_to(maf_out, c.maf, c.maf_bytes);
      }
    }
    pbsim_stats st;
    if (pbsim_cuda_simulate_end(eng, &st, nullptr, 0, nullptr) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    if (bam) {  // BGZF end-of-file marker (SAM spec 4.1.2)
      static const unsigned char eof[28] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43,
                                            0x02, 0, 0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0};
      reads_out.submit(reinterpret_cast<const char *>(eof), sizeof eof, true);
    }
    reads_out.close();
    maf_out.close();
    replay_pos += (size_t)st.res_pass_num;
    gen_seconds += st.gen_seconds;
    total_bases += st.res_len_total;
    return st;
  };
  auto print_stats_tail = [&](const pbsim_stats &st) {  // print_simulation_stats (:5551-5563)
    fprintf(stderr, "read length mean (SD) : %f (%f)\n", st.res_len_mean, st.res_len_sd);
    fprintf(stderr, "read length min : %ld\n", (long)st.res_len_min);
    fprintf(stderr, "read length max : %ld\n", (long)st.res_len_max);
    fprintf(stderr, "read accuracy mean (SD) : %f (%f)\n", st.res_accuracy_mean, st.res_accuracy_sd);
    fprintf(stderr, "substitution rate. : %f\n", (double)st.res_sub_num / st.res_len_total);
    fprintf(stderr, "insertion rate. : %f\n", (double)st.res_ins_num / st.res_len_total);
    fprintf(stderr, "deletion rate. : %f\n", (double)st.res_del_num / st.res_len_total);
    fprintf(stderr, "\n");
  };
  auto finish = [&]() {
    pbsim_cuda_destroy(eng);
    pbsim_host_model_free(hm);
    fprintf(stderr, ":::: System utilization ::::\n\n");
    fprintf(stderr, "CPU time(s) : %ld\n", now_cpu() - rst1);
    fprintf(stderr, "Elapsed time(s) : %ld\n", now_wall() - t1);
    fprintf(stderr, "\n:::: B200 engine ::::\n\n");
    fprintf(stderr, "input load time(s) : %.3f\n", load_seconds);
    fprintf(stderr, "waiting for record pieces (generation + device-to-host copies) (s) : %.3f\n", chunk_wait_seconds);
    fprintf(stderr, "copying gzip members into the output files (s) : %.3f (%.2f GB)\n", write_seconds, written_bytes / 1e9);
    fprintf(stderr, "generation device time(s) : %.3f\n", gen_seconds);
    fprintf(stderr, "simulated Gbp/s (generation only) : %.3f\n", gen_seconds > 0 ? total_bases / gen_seconds / 1e9 : 0.0);
    return 0;
  };

  if (!wgs) {
    // ---- main :760-868: the whole transcript table / template file is one run
    std::string ids;
    std::vector<int32_t> id_start{0};
    for (const std::string &id : S.ids) {
      ids += id;
      id_start.push_back((int32_t)ids.size());
    }
    pbsim_seqset ss;
    memset(&ss, 0, sizeof ss);
    ss.strategy = trans ? PBSIM_STRATEGY_TRANS : PBSIM_STRATEGY_TEMPL;
    ss.n = (int64_t)S.ids.size();
    ss.bases = S.bases.data();
    ss.start = S.start.data();
    ss.plus_exp = S.plus.data();
    ss.minus_exp = S.minus.data();
    ss.ids = ids.data();
    ss.id_start = id_start.data();
    memcpy(ss.hp_del_bias, bias, sizeof bias);
    if (pbsim_cuda_set_seqset(eng, &ss) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    if (o.hp_del_bias != 1) {  // the prepass of :2671-2746 / :3244-3310: expression-weighted homopolymer histogram
      int64_t f[12];
      pbsim_cuda_get_hpfreq(eng, f);
      pbsim_host_hp_del_bias(o.hp_del_bias, f, ss.hp_del_bias);
      if (pbsim_cuda_set_seqset(eng, &ss) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    }
    std::string sq;
    for (size_t t = 0; align && t < S.ids.size(); ++t)
      sq += "@SQ\tSN:" + S.ids[t] + "\tLN:" + std::to_string(S.start[t + 1] - S.start[t]) + "\n";
    const pbsim_stats st = simulate_to_files(o.prefix, o.id_prefix, 0, sq);
    fprintf(stderr, ":::: Simulation stats ::::\n\n");
    fprintf(stderr, "read num. : %ld\n", (long)st.res_num);
    print_stats_tail(st);
    return finish();
  }


  // ---- hp-del-bias (main :673-697)
  int64_t hp11_running = 0;
  auto seq_name = [&](size_t num) {  // RNAME / @SQ SN of sequence num: the first word of its FASTA header
    const std::string &id = seqs[num - 1].id;
    const size_t e = id.find_first_of(" \t\r\v\f");
    return id.substr(0, e);
  };
  auto ingest = [&](size_t num, const double b[12], int64_t hpfreq[12]) {
    // the split pass kept the text (identical to what genome_seq re-reads from <prefix>_NNNN.ref: the split writes
    // the body lines verbatim, :953-957)
    const std::string &seq = seqs[num - 1].text;
    pbsim_sequence s;
    s.bases = seq.data();
    s.len = (int64_t)seq.size();
    s.seq_num = (int32_t)num;
    memcpy(s.hp_del_bias, b, sizeof s.hp_del_bias);
    if (pbsim_cuda_set_sequence(eng, &s) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    if (align && pbsim_cuda_set_sequence_name(eng, seq_name(num).c_str()) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    pbsim_cuda_get_hpfreq(eng, hpfreq);
    return (int64_t)seq.size();
  };
  if (o.hp_del_bias != 1) {
    int64_t tot[12] = {0};
    for (size_t n = 1; n <= seqs.size(); ++n) {
      int64_t f[12];
      ingest(n, bias, f);
      for (int k = 0; k < 12; ++k) tot[k] += f[k];
    }
    hp11_running = tot[11];
    pbsim_host_hp_del_bias(o.hp_del_bias, tot, bias);
  }
  for (size_t n = 1; n <= seqs.size(); ++n) {
    int64_t f[12];
    const int64_t glen = ingest(n, bias, f);
    hp11_running += f[11];  // every process ingests every sequence: the aliased cell depends on all earlier ones
    if ((int)((n - 1) % (size_t)o.world) != o.rank) continue;
    double b[12];
    memcpy(b, bias, sizeof b);
    memcpy(&b[0], &hp11_running, sizeof(double));  // the cell genome.hpfreq[11] aliases in the reference build
    if (pbsim_cuda_update_hp_del_bias(eng, b) != 0) die("ERROR: %s\n", pbsim_cuda_last_error(eng));
    char stem[4096], pu[512];
    snprintf(stem, sizeof stem, "%s_%04zu", o.prefix.c_str(), n);
    snprintf(pu, sizeof pu, "%s%zu", o.id_prefix.c_str(), n);
    const std::string sq = align ? "@SQ\tSN:" + seq_name(n) + "\tLN:" + std::to_string(glen) + "\n" : "";
    const pbsim_stats st = simulate_to_files(stem, pu, (int64_t)(o.depth * glen), sq);  // sim.len_quota (:705)
    // print_simulation_stats (:5541-5564)
    fprintf(stderr, ":::: Simulation stats (ref.%zu) ::::\n\n", n);
    fprintf(stderr, "read num. : %ld\n", (long)st.res_num);
    fprintf(stderr, "depth : %lf\n", (double)st.res_len_total / glen / o.pass_num);
    print_stats_tail(st);
  }
  return finish();
}
