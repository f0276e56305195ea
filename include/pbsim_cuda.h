/* libpbsim_cuda — C ABI of the B200 read-generation engine.
 *
 * The reference (yukiteruono/pbsim3) has no plugin / FFI interface: the hot path is reached
 * through the internal seam  `int simulate_by_qshmm()` / `int simulate_by_errhmm()`
 * (src/pbsim.cpp:1955, :3594), called by main() once per reference sequence
 * (src/pbsim.cpp:699-754) and communicating through file-scope globals
 * (src/pbsim.cpp:184-197).  This header is that seam made explicit: every entry point
 * names the reference lines it replaces.  Plain pointers and sizes only.
 *
 *   host front end (pbsim_host_*)      replaces set_qshmm/set_errhmm/set_mut and the table
 *                                      builders inlined in simulate_by_* (host, runs once)
 *   engine         (pbsim_cuda_*)      replaces get_genome_seq's in-memory products, the
 *                                      read loop, the per-position chain, record emission
 *                                      and the statistics accumulation (GPU)
 *
 * All functions return 0 on success and a negative PBSIM_E_* code on failure;
 * pbsim_cuda_last_error() returns the message the reference would have printed (or a
 * CUDA error string).  One engine per GPU; calls on one engine come from one host thread.
 * There is no CPU fallback: if no CUDA device is usable pbsim_cuda_create fails.
 */
#ifndef PBSIM_CUDA_H
#define PBSIM_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 3: PBSIM_METHOD_SAMPLE, pbsim_cuda_set_pool, pbsim_host_sample_filter (additive over 2) */
#define PBSIM_ABI_VERSION 4

#define PBSIM_E_INVALID   (-1)  /* bad argument / call order                            */
#define PBSIM_E_CUDA      (-2)  /* CUDA runtime error                                   */
#define PBSIM_E_IO        (-3)  /* cannot open / parse a file                           */
#define PBSIM_E_PARAM     (-4)  /* "length/accuracy parameters are not appropriate"     */
#define PBSIM_E_REPLAY    (-5)  /* replay log exhausted or inconsistent with the run    */
#define PBSIM_E_OVERFLOW  (-6)  /* a read outgrew its scratch slot even after regrowth  */

#define PBSIM_METHOD_QSHMM  1   /* --method qshmm  (METHOD_QS,  pbsim.cpp:37) */
#define PBSIM_METHOD_ERRHMM 2   /* --method errhmm (METHOD_ERR, pbsim.cpp:38) */
#define PBSIM_METHOD_SAMPLE 3   /* --method sample (METHOD_SAM, pbsim.cpp:39): qualities copied from a pool of real reads */

#define PBSIM_RNG_PHILOX 0      /* Philox4x32-10 keyed by (seed, sequence, read id); engine-native */
#define PBSIM_RNG_REPLAY 1      /* consume a log of the reference's own rand() draws              */

#define PBSIM_STRATEGY_WGS   0   /* --strategy wgs   (STRATEGY_WGS,   pbsim.cpp:33) */
#define PBSIM_STRATEGY_TRANS 1   /* --strategy trans (STRATEGY_TRANS, pbsim.cpp:34) */
#define PBSIM_STRATEGY_TEMPL 2   /* --strategy templ (STRATEGY_TEMPL, pbsim.cpp:35) */

#define PBSIM_NQV 94            /* quality codes 0..93 (pbsim.cpp:191) */
#define PBSIM_NACC 101          /* accuracies 0..100  (ACCURACY_MAX, pbsim.cpp:42) */

/* ------------------------------------------------------------------------------------------
 * Quantised model: exactly the integer lookup tables the reference builds at the top of every
 * simulate_by_* call, 0-based (table[k] here is the reference's table[k+1]).
 * ---------------------------------------------------------------------------------------- */

/* one accuracy row of the HMM tables.
 * qshmm : init2state / emis2qc / tran2state, resolution 100  (pbsim.cpp:2066-2144)
 *         or, when the model has no such accuracy, freq2qc, resolution 1000 (:2145-2169)
 * errhmm: init2state / emis2err / emis2del / tran2state, resolution 1000 (:3708-3789) */
typedef struct {
  int32_t exists;          /* exist_hmm[acc]                                              */
  int32_t nstates;         /* rows 1..nstates are valid (row 0 unused)                    */
  int32_t resolution;      /* row stride of tran[] / emis[]: 100 or 1000                  */
  int32_t init_mod;        /* qc_rand_value_init / err_rand_value_init                    */
  const uint8_t *init;     /* [init_mod] -> state                                         */
  const int32_t *tran_mod; /* [nstates+1] row modulus                                     */
  const uint8_t *tran;     /* [(nstates+1)*resolution] -> next state                      */
  const int32_t *emis_mod; /* [nstates+1]                                                 */
  const uint8_t *emis;     /* [(nstates+1)*resolution] -> QV (qshmm) | 0,1,2 (errhmm)     */
  const int32_t *emis_del; /* errhmm: emis2del[state] on the 1..1000 scale, else NULL     */
  int32_t freq_mod;        /* qshmm without model: qc_rand_value_freq                     */
  const uint8_t *freq;     /* [freq_mod] -> QV                                            */
} pbsim_hmm_row;

typedef struct {
  int32_t method;                  /* PBSIM_METHOD_*                                         */
  int32_t pass_num;                /* --pass-num                                             */
  int64_t len_min, len_max;        /* --length-min/max                                       */
  double accuracy_mean;            /* after set_sim_param truncation; printed as rq:f (:2333) */
  char id_prefix[128];             /* --id-prefix                                            */
  /* length / accuracy samplers (pbsim.cpp:1991-2064) */
  const int32_t *prob2len;         /* [len_rand_value]                                       */
  int32_t len_rand_value;
  const uint8_t *prob2accuracy;    /* [accuracy_rand_value]                                  */
  int32_t accuracy_rand_value;
  int32_t acc_lo, acc_hi;          /* accuracy_min / accuracy_max the sampler can return     */
  /* set_mut thresholds on the 0..999999 scale (pbsim.cpp:5474-5479) and Phred probs (:546) */
  int32_t sub_thre[PBSIM_NQV], ins_thre[PBSIM_NQV], del_thre[PBSIM_NQV];
  double qc_prob[PBSIM_NQV];
  /* HMM */
  int32_t model_acc_min, model_acc_max; /* errhmm.acc_min / acc_max (pbsim.cpp:5665-5678)    */
  pbsim_hmm_row rows[PBSIM_NACC];
} pbsim_model;

/* one reference sequence as get_genome_seq leaves it (pbsim.cpp:997-1068) */
typedef struct {
  const char *bases;       /* ASCII, any case (upper-cased on the device like :1035-1037)   */
  int64_t len;
  int32_t seq_num;         /* genome.num, 1-based; part of read ids and of the Philox key   */
  double hp_del_bias[12];  /* genome.hp_del_bias[0..10] plus the two cells the reference    *
                            * reads out of bounds ([0] for hp[-1], [11] for runs >= 11)     */
} pbsim_sequence;

/* a set of sequences simulated in one run: the transcript table of --strategy trans as
 * get_transcript_inf and the fgets loops of simulate_by_*_trans read it (pbsim.cpp:1075-1140,
 * :2748-2772), or the template FASTA of --strategy templ (:1366-1417, :3312-3329).  The caller
 * parses the file; sequences arrive concatenated.  Reads are numbered 1.. through the whole set
 * (sim.res_num): transcript t yields plus_exp[t] '+' reads then minus_exp[t] '-' reads, each a
 * window of it (length, accuracy and start position drawn, :2842-2866); a template yields one
 * '+' read covering it (:3359-3364). */
typedef struct {
  int32_t strategy;          /* PBSIM_STRATEGY_TRANS or PBSIM_STRATEGY_TEMPL                  */
  int64_t n;                 /* sequences                                                     */
  const char *bases;         /* concatenated text, case as in the file                        */
  const int64_t *start;      /* [n+1] offsets into bases; total < 2^32 - 2^16                 */
  const int32_t *plus_exp;   /* [n] trans only (may be NULL for templates)                    */
  const int32_t *minus_exp;  /* [n]                                                           */
  const char *ids;           /* concatenated names (transcript.id / templ.id, <= 128 chars)   */
  const int32_t *id_start;   /* [n+1]                                                         */
  double hp_del_bias[12];    /* transcript.hp_del_bias / templ.hp_del_bias, cells as above    */
} pbsim_seqset;

typedef struct {
  int32_t rng_mode;              /* PBSIM_RNG_*                                              */
  uint32_t seed;                 /* --seed                                                   */
  int64_t len_quota;             /* sim.len_quota = depth * genome.len (pbsim.cpp:705)       */
  int64_t first_read;            /* number of reads already simulated for this sequence      *
                                  * (0 for a whole-sequence run; >0 when read-id ranges are  *
                                  * sharded across GPUs)                                     */
  int64_t len_total_start;       /* emitted bases of those earlier reads                     */
  int64_t max_reads;             /* stop after this many reads even if the quota is not met  *
                                  * (0 = run to the quota)                                   */
  int64_t batch_reads;           /* reads per chunk (0 = engine default)                     */
  /* replay mode: the reference's draw stream and where every (read, pass) starts in it */
  const int32_t *replay_draws;
  int64_t replay_ndraws;
  const int64_t *replay_starts;  /* [replay_nsubreads]                                       */
  int64_t replay_nsubreads;
} pbsim_run;

/* a chunk = the records of a contiguous range of reads, in read order, exactly the bytes the
 * reference fprintf()s to fp_fq|fp_sam and fp_maf (pbsim.cpp:2318-2383) */
typedef struct {
  const char *reads;        /* FASTQ (pass_num == 1) or SAM records (no @HD/@RG header)      */
  int64_t reads_bytes;
  const char *maf;          /* MAF blocks, or with option "align" SAM alignment lines (no header), or with
                             * "align_bam" BAM alignment records (no BAM header; with "deflate", BGZF blocks) */
  int64_t maf_bytes;
  int64_t first_read, n_reads;   /* 1-based id of the first read, number of reads            */
  int64_t bases;                 /* emitted read bases in this chunk, all passes             */
  int32_t on_device;             /* 1: pointers are device pointers                          */
  int32_t compressed;            /* 1: option "deflate": the bytes are gzip members (host    *
                                  * delivery only); concatenated they gunzip to the text     */
  int64_t reads_text_bytes;      /* text size of the batch's records (set with first_read)   */
  int64_t maf_text_bytes;
} pbsim_chunk;

/* sim.res_* (pbsim.cpp:63-70) after the run; histograms are freq_len / freq_accuracy (:195-196) */
typedef struct {
  int64_t res_num, res_pass_num;
  int64_t res_len_total;
  int64_t res_len_min, res_len_max;
  int64_t res_sub_num, res_ins_num, res_del_num;
  double accuracy_total;         /* running sum of per-read accuracies, in read order        */
  double res_len_mean, res_len_sd;
  double res_accuracy_mean, res_accuracy_sd;
  double gen_seconds;            /* device time of all generation steps (CUDA events)        */
  double sim_seconds;            /* ... of which pass 1 (k_sim_qshmm / k_sim_errhmm)          */
  double emit_seconds;           /* ... of which pass 2 (k_emit)                             */
  double deflate_seconds;        /* ... of which the gzip writer (option "deflate")          */
  double seg_seconds;            /* ... of which the segment kernel (k_sim_seg / _err) alone  */
  int64_t kernel_launches;       /* number of engine kernels launched during the run         */
  double chain_seconds;          /* ... of which the chain-chunk kernel (k_qs_pass1 / k_chain_chunk_err) alone (ABI 4) */
  int64_t len_total_end;         /* the quota counter when the run ended: len_total_start + the bases this run's *
                                  * reads emitted in pass 0 (:2297) = len_total_start of the next read range (ABI 4) */
} pbsim_stats;

typedef struct pbsim_engine pbsim_engine;

/* ------------------------------------------------------------------------------------------
 * engine
 * ---------------------------------------------------------------------------------------- */
int pbsim_cuda_abi_version(void);
const char *pbsim_cuda_last_error(const pbsim_engine *e); /* e may be NULL: last create error */

int pbsim_cuda_create(pbsim_engine **out, int device);
void pbsim_cuda_destroy(pbsim_engine *e);

/* replaces: the static tables of simulate_by_qshmm/errhmm + set_mut (host -> device upload).
 * The pbsim_model (and the tables it points to) must stay alive while the engine uses it. */
int pbsim_cuda_set_model(pbsim_engine *e, const pbsim_model *m);

/* replaces: get_genome_seq's genome.seq / genome.hp (pbsim.cpp:1032-1065): uploads the ASCII
 * sequence, upper-cases, computes homopolymer lengths, packs to 2 bits per base */
int pbsim_cuda_set_sequence(pbsim_engine *e, const pbsim_sequence *s);
/* RNAME of the alignment lines of the current WGS sequence (option "align"); required before simulate_begin then
 * (not with "align_bam", whose records name the sequence by refID 0).
 * set_sequence and set_synthetic_sequence forget it.  1 to 4096 printable characters, no whitespace. */
int pbsim_cuda_set_sequence_name(pbsim_engine *e, const char *name);
/* replaces: the per-sequence ingest of simulate_by_{qshmm,errhmm}_{trans,templ} (upper-casing with the
 * reference's first-base quirk, homopolymer lengths per sequence) for a whole set at once; needs set_model
 * first (which of the four functions is restated depends on the method).  After it, simulate_begin runs
 * the set: pbsim_run.len_quota is ignored, first_read / max_reads select a range of read numbers.
 * get_hpfreq then returns the expression-weighted histogram of the --hp-del-bias prepass (:2671-2746). */
int pbsim_cuda_set_seqset(pbsim_engine *e, const pbsim_seqset *s);
/* --method sample: the pool get_sample_inf leaves in fp_filtered (pbsim.cpp:1214-1275) — the quality strings of
 * the sample reads that pass the length and accuracy filters, in file order, concatenated (quals, qstart[n+1]).
 * The caller parses and filters the FASTQ (host front end: pbsim_host_sample_filter).  A run with a model of
 * method PBSIM_METHOD_SAMPLE then replaces simulate_by_sample (:1694-1949): every read copies the qualities of a
 * pool entry; the copies of one entry follow each other and each is as long as the previous copy's read (:1756,
 * :1835).  Single-pass, --strategy wgs only, whole sequences only (first_read = max_reads = 0). */
int pbsim_cuda_set_pool(pbsim_engine *e, const char *quals, const int64_t *qstart, int64_t n);
/* synthetic i.i.d. ACGT sequence generated on the device (benchmarks; no host transfer) */
int pbsim_cuda_set_synthetic_sequence(pbsim_engine *e, int64_t len, int32_t seq_num, uint64_t seed);
/* replace hp_del_bias of the current sequence without re-ingesting it (bias[0] is only known once the
 * sequence's own hpfreq[11] is, see pbsim_host_hp_del_bias); the set of cells equal to 1 must not change */
int pbsim_cuda_update_hp_del_bias(pbsim_engine *e, const double hp_del_bias[12]);
/* upper-cased text of the current sequence (tests, benchmarks) */
int pbsim_cuda_get_sequence_ascii(pbsim_engine *e, char *dst, int64_t cap);
/* device products of the last set_sequence / set_seqset / set_synthetic_sequence (tests): pk[ceil(len/16)] 2-bit
 * codes (A=0 C=1 G=2 T=3, base i at bits 2*(i%16) of word i/16), hp4[ceil(len/2)] 4-bit homopolymer lengths (base i
 * in the low nibble of byte i/2 when i is even), xm[ceil(ceil(len/1024)/32)] exceptional-block bits (block b at bit
 * b%32 of word b/32).  len must be the current sequence's length. */
int pbsim_cuda_get_sequence_tables(pbsim_engine *e, uint32_t *pk, uint8_t *hp4, uint32_t *xm, int64_t len);
/* homopolymer histogram of the current sequence, genome.hpfreq[0..10] plus the aliased [11] */
int pbsim_cuda_get_hpfreq(pbsim_engine *e, int64_t hpfreq[12]);

/* replaces: one simulate_by_qshmm() / simulate_by_errhmm() call for the current sequence */
int pbsim_cuda_simulate_begin(pbsim_engine *e, const pbsim_run *run);
/* 1: chunk filled, 0: finished.  Host delivery: the records of a batch of reads stay in HBM and are
 * handed out as consecutive PIECES of at most `stage_bytes` per stream through double-buffered pinned
 * staging (pointers valid until the next call); concatenating the pieces gives the byte streams in
 * read order.  first_read / n_reads / bases are set on the first piece of every batch. */
int pbsim_cuda_next_chunk(pbsim_engine *e, pbsim_chunk *c);
/* same, records stay in HBM (c->on_device = 1) */
int pbsim_cuda_next_chunk_device(pbsim_engine *e, pbsim_chunk *c);
/* stats; freq_len has len_max*2+2 cells, freq_accuracy 100001; either may be NULL */
int pbsim_cuda_simulate_end(pbsim_engine *e, pbsim_stats *st, int64_t *freq_len, int64_t freq_len_cells,
                            int64_t *freq_accuracy);
/* CUDA-event timer on the engine's stream: stop=0 records the start, stop=1 records the stop,
 * waits for it and returns the elapsed device milliseconds */
int pbsim_cuda_device_timer(pbsim_engine *e, int stop, double *ms);
/* tunables: "stage_bytes" (pinned staging per stream and slot, default 128 MiB),
 * "target_batch_bases" (emitted bases per batch of reads, default 6 Gi),
 * "segments" (1: segment-parallel pass 1 for long reads in PHILOX mode, default 1; results are identical
 * either way), "seg_min_len" (shortest read that is segmented, default 2048), "chain_chunk" (segments one thread of the
 * chain / quality pass walks; 0 (default): by method — 8 for qshmm, 32 for errhmm; results are identical for any value),
 * "pipeline" (0: batches are generated inside next_chunk; 1 (default): with host delivery a producer thread
 * generates batch k+1 into a second record buffer while batch k is handed out; 2: also for device delivery),
 * "host_batch_bases" (batch size of pipelined host delivery, default 1 Gi),
 * "deflate" (1: host delivery hands out gzip members written on the GPU — every 32 KiB of a record stream is one
 * member holding up to eight dynamic-Huffman blocks of literals — instead of text: what the reference's `gzip >` children produce,
 * pbsim.cpp:708-730; default 0),
 * "bam" (1: with pass_num > 1 the reads stream holds BAM alignment records — the binary form of the reference's SAM
 * lines, what its `samtools view -b` child writes (pbsim.cpp:715-722) — and, with "deflate", BGZF blocks; the caller
 * adds the BAM header block in front and the BGZF end-of-file block behind; default 0),
 * "align" (1: the second stream holds one SAM alignment line per (read, pass) instead of its MAF block: QNAME as in
 * the reads stream, FLAG 0 / 16 (4: no match or substitution column), RNAME (WGS: pbsim_cuda_set_sequence_name; sets:
 * the sequence's id), 1-based POS, MAPQ 60, CIGAR of =, X, I, D in reference order (insertions in front of the first
 * and behind the last = / X column become S, deletions there are dropped), RNEXT * PNEXT 0 TLEN 0, SEQ and QUAL in
 * reference orientation, NM:i; no header lines; not with "bam" unless "align_bam"; default 0),
 * "align_bam" (1, needs "align": the second stream holds one BAM alignment record (SAM spec 4.2) per (read, pass)
 * instead, which decodes to exactly the SAM line "align" writes: refID 0 for WGS (the caller's one @SQ), the sequence's
 * index in the set for sets, -1 unmapped; pos = POS - 1; MAPQ 60 (unmapped 0); bin = reg2bin(pos, pos + the =, X, D
 * columns) (unmapped 4680); CIGAR ops = 7, X 8, I 1, D 2, S 4; next refID -1, next pos -1, tlen 0; SEQ as 4-bit codes
 * high nibble first, the odd pad nibble 0; QUAL values; tag NM of type C, S or I by size.  A record of more than
 * 65,535 ops holds the two ops <l_seq>S<span>N in its CIGAR field and the real ops in a CG:B:I tag behind NM (SAM spec
 * 4.2.2).  With "deflate" the records travel as BGZF blocks; the caller writes the BAM header (magic, header text,
 * n_ref, the references in @SQ order) in front and the BGZF end-of-file block behind.  With "bam" (pass_num > 1)
 * both streams are BAM.  maf_text_bytes counts the record bytes; default 0),
 * "sample_spec" (--method sample; 1 (default): every copy of a pool entry is first simulated in its own thread at
 * the entry's length and only the copies that follow a shorter read are redone as chains; 0: one thread walks all
 * copies of an entry; results are identical either way; with "segments" the speculative pass of reads of at least
 * "seg_min_len" positions runs on the segment kernels) */
int pbsim_cuda_set_option(pbsim_engine *e, const char *name, int64_t value);
/* device pointer + cell count of the int64 stats block {counters[16], freq_accuracy[100001],
 * freq_len[2*len_max+2]} so that a multi-GPU driver can ncclAllReduce it in place */
int pbsim_cuda_stats_device_block(pbsim_engine *e, void **dptr, int64_t *cells);

/* debugging / tests: per-(read, pass) results of the last chunk, 8 int64 per subread:
 * {read_id, pass, acc, offset, wlen, rlen, ncol, strand} */
int pbsim_cuda_last_chunk_info(pbsim_engine *e, int64_t *out, int64_t cap_subreads, int64_t *n_subreads);

/* ------------------------------------------------------------------------------------------
 * host front end (no GPU needed)
 * ---------------------------------------------------------------------------------------- */
typedef struct pbsim_host_model pbsim_host_model;

/* sim_t subset that shapes the tables; accuracy_mean must already be truncated like
 * set_sim_param does (pbsim.cpp:1660) */
typedef struct {
  int32_t method;
  int32_t pass_num;
  int64_t len_min, len_max;
  double len_mean, len_sd;
  double accuracy_mean;
  int64_t sub_ratio, ins_ratio, del_ratio;
  char id_prefix[128];
} pbsim_host_params;

/* replaces set_qshmm / set_errhmm (pbsim.cpp:5570-5714) + set_mut (:5471) + the table builders
 * (:1991-2170, :3633-3789).  On failure *err (if not NULL) receives a static message. */
int pbsim_host_model_load(pbsim_host_model **out, const pbsim_host_params *p, const char *model_path,
                          const char **err);
const pbsim_model *pbsim_host_model_get(const pbsim_host_model *m);
void pbsim_host_model_free(pbsim_host_model *m);

/* main()'s --hp-del-bias handling (pbsim.cpp:673-697): hpfreq accumulated over all sequences ->
 * bias[1..10]; bias[0]/bias[11] are the out-of-bounds cells (see DESIGN.md "reference quirks") */
/* the "sequencing start pos distribution" of --strategy trans (pbsim.cpp:2504-2528): for rank 1..rank_max,
 * ends[rank*21 + j] = last table position (1..1000) of start fraction 5*j percent, 0xFFFF after the row
 * ended; mod[rank] = ssp_rand_value[rank].  ends has (rank_max+1)*21 cells, mod rank_max+1. */
void pbsim_host_ssp_table(int32_t rank_max, uint16_t *ends, uint16_t *mod);
/* the literal code (bit-reversed code | length << 16 for bytes 0..255, then end-of-block) and the DEFLATE dynamic
 * block header (LSB-first bit string) the engine's gzip writer derives from a stream's byte histogram */
int pbsim_host_deflate_code(const int64_t hist[256], uint32_t lit[257], uint32_t *hdr_bits, uint32_t *hdr_words,
                            int32_t cap_words);
/* get_sample_inf (pbsim.cpp:1155-1330) over a FASTQ held in memory: every 4th '\n'-terminated line is a quality
 * string (a last line without line feed is not counted, like fgets + trim do); strings whose length lies in
 * [len_min, len_max] and whose accuracy 1 - mean(10^(-q/10)) lies in [accuracy_min, accuracy_max] are appended to
 * quals (capacity: bytes) in file order, qstart[0..*n_out] are their offsets (capacity qstart_cap cells).
 * st receives the numbers print_sample_stats shows (:1336-1358) and the sample profile stores (:1317-1326).
 * Errors carry the reference's message in *err. */
typedef struct {
  int64_t num, len_total, len_min, len_max;                                         /* all reads      */
  int64_t num_filtered, len_total_filtered, len_min_filtered, len_max_filtered;     /* filtered reads */
  double len_mean_filtered, len_sd_filtered, accuracy_mean_filtered, accuracy_sd_filtered;
} pbsim_sample_stats;
int pbsim_host_sample_filter(const char *fastq, int64_t bytes, int64_t len_min, int64_t len_max, double accuracy_min,
                             double accuracy_max, char *quals, int64_t *qstart, int64_t qstart_cap, int64_t *n_out,
                             pbsim_sample_stats *st, const char **err);
void pbsim_host_hp_del_bias(double hp_del_bias_opt, const int64_t hpfreq[12], double bias[12]);

#ifdef __cplusplus
}
#endif
#endif
