#!/usr/bin/env python
"""bench.py — simulated Gbp/s of the PBSIM3 read-generation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c1|c2|c4|c5|cs] [--impl reference]
                    [--dump-outputs DIR]

A STEP is one call of the reference's seam for one reference sequence: ingest the sequence
(get_genome_seq), then simulate_by_qshmm / simulate_by_errhmm to the depth quota, records emitted
(FASTQ + MAF).  Sequences are the 24 contigs of a synthetic 3.1 Gbp human-sized genome; the timed steps are the
sequences (warmup + k) mod 24.  With N GPUs the steps are ONE run split over the ranks: the line of all their reads
is cut into N pieces of equal estimated work (whole sequences plus read ranges of the sequences two ranks share).
Default workload "c3" = BASELINE.json configs[2] (WGS qshmm, QSHMM-ONT ultra-long reads, 3.1 Gbp genome, --depth 50):
the configuration the metric "simulated Gbp/s (WGS qshmm, 3.1 Gbp genome)" is quoted on.

  value    : emitted bases / device time, sequence text already resident in HBM, records left in HBM; two engines per
             GPU work on alternate sequences (--lanes)
  e2e      : same steps through the C ABI with HOST buffers: the sequence text is uploaded from pinned host memory and
             every record byte is delivered to pinned host memory inside the timed region, as gzip members written by
             the GPU — the reference's output files are .fq.gz / .maf.gz (pbsim.cpp:708-730)
  e2e_text : the same delivering the uncompressed text (4.1 bytes per base over PCIe instead of 1.6)
  roofline / cpu_baseline : see DESIGN.md "Measurement"

--impl reference times the UNMODIFIED reference binary (oracle/_ref/pbsim, compiled from
/root/reference/src/pbsim.cpp by `make -C oracle ref`) on the host cores, as N seed-split processes.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# GRCh38-like contig sizes (Mbp), total 3.088 Gbp, every sequence < 250 Mbp (reference limit 1e9, pbsim.cpp:24)
CONTIG_MBP = [248, 242, 198, 190, 182, 171, 159, 145, 138, 134, 135, 133, 114, 107, 102, 90, 83, 80, 59, 64, 47,
              51, 156, 57]
GENOME_SEED = 20240501

WORKLOADS = {
    # BASELINE.json configs[2]
    "c3": dict(name="WGS qshmm QSHMM-ONT ultra-long (mean 50 kb), 3.1 Gbp synthetic genome, --depth 50",
               method="qshmm", model="QSHMM-ONT.model", depth=50.0,
               params=dict(len_mean=50000.0, len_sd=35000.0, len_max=1000000, ratio=(39, 24, 36)),
               cli=["--length-mean", "50000", "--length-sd", "35000", "--length-max", "1000000",
                    "--difference-ratio", "39:24:36"]),
    # configs[0]'s model and defaults on the named genome size
    "c1": dict(name="WGS qshmm QSHMM-RSII defaults (mean 9 kb), 3.1 Gbp synthetic genome, --depth 20",
               method="qshmm", model="QSHMM-RSII.model", depth=20.0, params=dict(), cli=[]),
    # configs[1]
    "c2": dict(name="WGS errhmm ERRHMM-ONT-HQ (mean 9 kb), 3.1 Gbp synthetic genome, --depth 30",
               method="errhmm", model="ERRHMM-ONT-HQ.model", depth=30.0, params=dict(), cli=[]),
    # configs[4]: multi-pass CLR, SAM records (pbsim.cpp:2322-2333) instead of FASTQ
    "c5": dict(name="WGS errhmm ERRHMM-SEQUEL --pass-num 10 (mean 9 kb), 3.1 Gbp synthetic genome, --depth 20, SAM+MAF",
               method="errhmm", model="ERRHMM-SEQUEL.model", depth=20.0, params=dict(pass_num=10),
               cli=["--pass-num", "10"], batch_bases=3 << 30),
    # --method sample (SURVEY 8f-2): qualities copied from a pool of real reads; the pool is made the way a user would make
    # it (reads simulated with QSHMM-RSII, filtered by pbsim_host_sample_filter)
    "cs": dict(name="WGS --method sample (pool: simulated QSHMM-RSII reads of a 30 Mbp sequence x 20, mean 9 kb), 3.1 Gbp "
                    "synthetic genome, --depth 20",
               method="sample", model=None, depth=20.0, params=dict(), cli=[]),
    # configs[3]: transcriptome; a step is one run over the whole transcript table
    "c4": dict(name="trans qshmm QSHMM-RSII, 200,000 synthetic transcripts (log-normal, median 1.5 kb), Zipf "
                    "expression, 2e7 reads",
               method="qshmm", model="QSHMM-RSII.model", depth=0.0, params=dict(), cli=[], strategy="trans",
               n_transcripts=200000, n_reads=20000000),
}

# algorithmic bytes per emitted base (SURVEY.md §8d): FASTQ 2.002 + MAF 2.122 written + 0.244 read (2-bit genome)
ALGO_BYTES_PER_BASE = 4.37


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (recipe in B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.path = os.path.join(tempfile.gettempdir(), "pbsim_clocks_%d_%d.csv" % (os.getpid(), gpu_index))
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, smax, reasons = [], [], set()
        try:
            with open(self.path) as f:
                for line in f:
                    p = [x.strip() for x in line.split(",")]
                    if len(p) < 9:
                        continue
                    try:
                        sm.append(float(p[1]))
                        smax.append(float(p[2]))
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                       p[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference binary on the host cores
# ------------------------------------------------------------------------------------------------
def _ref_sample_genome(path, mbp=5):
    import numpy as np
    rng = np.random.default_rng(GENOME_SEED)
    s = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=mbp * 1000000)].tobytes()
    with open(path, "wb") as f:
        f.write(b">sample\n")
        for i in range(0, len(s), 70):
            f.write(s[i:i + 70] + b"\n")
    return len(s)


def _parse_ref_bases(stderr):
    total = 0
    num = None
    for line in stderr.splitlines():
        if line.startswith("read num. :"):
            num = int(line.split(":")[1])
        elif line.startswith("read length mean (SD) :") and num is not None:
            total += int(round(num * float(line.split(":")[1].split("(")[0])))
            num = None
    return total


def run_reference_processes(wl, nproc, depth, workdir, seed0=1):
    """Launch nproc seed-split reference processes (--seed s+i) on the sample genome; returns (bases, wall)."""
    from oracle import refrun as R
    from tests.golden_util import model_path
    fa = os.path.join(workdir, "sample.fa")
    if not os.path.exists(fa):
        _ref_sample_genome(fa)
    env = dict(os.environ)
    env["PATH"] = R.SHIMS + ":" + env.get("PATH", "")  # gzip -> cat: generation + text formatting only
    args = ["--strategy", "wgs", "--method", wl["method"], "--" + wl["method"], model_path(wl["model"]),
            "--genome", fa, "--depth", str(depth)] + wl["cli"]
    procs = []
    t0 = time.perf_counter()
    for i in range(nproc):
        d = os.path.join(workdir, "p%d" % i)
        os.makedirs(d, exist_ok=True)
        procs.append(subprocess.Popen([R.REF_BIN] + args + ["--seed", str(seed0 + i), "--prefix", "o"], cwd=d, env=env,
                                      stdout=subprocess.DEVNULL, stderr=subprocess.PIPE))
    bases = 0
    for p in procs:
        _, err = p.communicate()
        bases += _parse_ref_bases(err.decode(errors="replace"))
    wall = time.perf_counter() - t0
    for i in range(nproc):
        d = os.path.join(workdir, "p%d" % i)
        for fn in os.listdir(d):
            try:
                os.remove(os.path.join(d, fn))
            except OSError:
                pass
    return bases, wall


def cpu_baseline(wl, kind_wanted="reference"):
    """Single-process reference on a bounded sample (about 10-20 s of CPU work)."""
    from oracle import refrun as R
    work = tempfile.mkdtemp(prefix="pbsim_cpu_")
    if R.have_reference_binary():
        depth = 24
        bases, wall = run_reference_processes(wl, 1, depth, work)
        return {"value": bases / wall / 1e9, "unit": "Gbp/s", "cores": 1, "kind": "reference",
                "sample": "unmodified reference binary (g++ -O2), 1 process, 5 Mbp synthetic contig, --depth %d "
                          "(%d bases in %.1f s), gzip children replaced by cat (generation + formatting only)"
                          % (depth, bases, wall)}
    # the reference binary did not travel: time the C restatement instead
    from oracle import oracle as O
    from tests.golden_util import model_path
    import numpy as np
    o = O.Oracle(wl["method"], model_path(wl["model"]), **wl["params"])
    o.rng_glibc(1)
    rng = np.random.default_rng(GENOME_SEED)
    s = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=5000000)].tobytes()
    o.set_sequence(s, 1)
    t0 = time.perf_counter()
    _, _, st = o.simulate_wgs(12)
    wall = time.perf_counter() - t0
    return {"value": st.res_len_total / wall / 1e9, "unit": "Gbp/s", "cores": 1, "kind": "port",
            "sample": "oracle C restatement, 5 Mbp synthetic contig, --depth 12 (%d bases in %.1f s)"
                      % (st.res_len_total, wall)}


def reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if wl["method"] == "sample":
        print(json.dumps({"impl": "reference", "unavailable": "the reference arm is set up for the qshmm / errhmm workloads"}))
        return
    from oracle import refrun as R
    base = {"impl": "reference", "metric": "simulated Gbp/s", "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic", "config": make_config(wl, args, args.gpus)}
    if not R.have_reference_binary():
        cb = cpu_baseline(wl)
        base.update(value=cb["value"], ms_per_step=None, cpu_baseline=cb,
                    e2e={"value": cb["value"], "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        print(json.dumps(base))
        return
    nproc = os.cpu_count() or 1
    work = tempfile.mkdtemp(prefix="pbsim_refarm_")
    depth = 3  # per process and step: 5 Mbp x 3 = 15 Mbase, a couple of seconds
    for w in range(args.warmup):
        run_reference_processes(wl, nproc, depth, work, seed0=1000 + w * nproc)
    tot_b, tot_t = 0, 0.0
    for k in range(args.steps):
        b, t = run_reference_processes(wl, nproc, depth, work, seed0=1 + k * nproc)
        tot_b += b
        tot_t += t
    v = tot_b / tot_t / 1e9
    base.update(value=v, ms_per_step=tot_t / max(1, args.steps) * 1e3,
                cpu_baseline={"value": v, "unit": "Gbp/s", "cores": nproc, "kind": "reference",
                              "sample": "unmodified reference binary, %d seed-split processes per step, each 5 Mbp "
                                        "synthetic contig --depth %d; gzip children replaced by cat" % (nproc, depth)},
                e2e={"value": v, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(base))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of ONE launch of the three big kernels on the c3 workload,
# and the read positions that launch covered, from the committed ncu captures (profiles/r02_k_*_c3_final.txt)
NCU_DRAM_BYTES = {
    # one batch of 128,851 reads: 6,565,276 segments = 6.72e9 simulated positions, 6.34e9 emitted bases
    "k_chain_chunk": dict(bytes=16.81e9, positions=6.72e9, src="profiles/r02_k_chain_chunk_c3_final.txt"),
    "k_sim_seg": dict(bytes=27.96e9, positions=6.72e9, src="profiles/r02_k_sim_seg_c3_final.txt"),
    "k_emit_rows": dict(bytes=41.26e9, positions=6.34e9, src="profiles/r02_k_emit_rows_c3_final.txt"),
}
# algorithmic bytes per read position of each kernel: the quality pass writes a 2-byte slot entry per position; the
# error pass reads and rewrites it; the row kernel reads it and 0.244 B of 2-bit genome and writes the records (4.124 B)
KERNEL_ALGO_BYTES = {"k_chain_chunk": 2.0, "k_sim_seg": 4.0, "k_emit_rows": 2.0 + 0.244 + 4.124}


def make_config(wl, args, world):
    """static description of the workload: identical in both arms (ours and --impl reference)"""
    trans = wl.get("strategy") == "trans"
    contigs = [max(200000, int(m * 1000000 * args.scale)) for m in CONTIG_MBP]
    if trans:
        sharding = ("strong scaling: the read numbers of the set are split into %d contiguous ranges (no quota in this "
                    "strategy); one NCCL all-reduce of the statistics block" % world)
    elif getattr(args, "no_split", False) or world == 1:
        sharding = ("strong scaling: the %d sequences of the timed steps are assigned to the ranks longest-first (LPT), "
                    "each simulated whole by one rank to its own depth quota; no data-path collective, one NCCL "
                    "all-reduce of the statistics block" % args.steps)
    else:
        sharding = ("strong scaling: ONE run of %d sequences, each to its own depth quota; the line of all their reads is "
                    "cut into %d pieces of equal estimated work (a rank owns whole sequences plus at most one leading "
                    "and one trailing read range of a sequence shared with a neighbour); results depend only on (seed, "
                    "sequence, read number), so the parts concatenate to the 1-GPU bytes; the quota cut of a shared "
                    "sequence takes the emitted bases of its earlier parts from one asynchronous NCCL all-reduce (an "
                    "int64 per sequence), plus one NCCL all-reduce of the statistics block" % (args.steps, world))
    return {"workload": wl["name"],
            "step": ("one run over the transcript table, FASTQ+MAF emitted" if trans else
                     "one reference sequence: ingest + simulate to depth quota, %s+MAF emitted"
                     % ("SAM" if wl["params"].get("pass_num", 1) > 1 else "FASTQ")),
            "genome_bp": int(sum(contigs)) if not trans else None, "contigs": len(contigs) if not trans else 1,
            "rng": "philox4x32-10 (ours) / libc rand() (reference)",
            "l2": "every step writes > 10 GB of records and events (>> 126 MB L2); no explicit flush needed",
            "scale": args.scale, "sharding": sharding,
            "engines_per_gpu": ("%d: every GPU runs %d engines, each driven by its own host thread on alternate sequences, so "
                                "that kernels bound by different things (shared-memory latency, instruction issue, HBM) "
                                "overlap" % (args.lanes, args.lanes)) if args.lanes > 1 else "1"}


def host_d2h_ceiling(barrier, allsum, reps=8, nbytes=256 << 20):
    """what the delivery path can reach at best on THIS box: aggregate GB/s of bare device -> pinned host copies issued
    by all ranks at once (measured in this run; tools/d2h_ceiling.py is the stand-alone version, its numbers for the
    pool's 8-GPU host are in profiles/r02_d2h_ceiling_8gpu.json)"""
    import torch
    try:
        d = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        h.copy_(d, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            h.copy_(d, non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        mine = nbytes * reps / dt / 1e9
        return allsum(mine), mine
    except Exception:
        return None, None


def lpt_assign(sizes, world):
    from pbsim_b200.stats_reduce import lpt_assign as f
    return f(sizes, world)


class Workload:
    """one engine set up for one BASELINE.json configuration"""

    def __init__(self, key, args, local, rank, overrides=True):
        import numpy as np
        from pbsim_b200 import capi, simulator
        from tests.golden_util import model_path
        self.np, self.capi = np, capi
        wl = dict(WORKLOADS[key])
        if overrides and (args.len_sd is not None or args.len_mean is not None):
            wl["params"] = dict(wl["params"])
            if args.len_sd is not None:
                wl["params"]["len_sd"] = args.len_sd
            if args.len_mean is not None:
                wl["params"]["len_mean"] = args.len_mean
            wl["name"] += " [diagnostic override: len_mean=%s len_sd=%s]" % (args.len_mean, args.len_sd)
        self.wl, self.key, self.rank = wl, key, rank
        L = capi.load()
        self.pool = None
        if wl["method"] == "sample":
            pe = simulator.Engine(local)
            pe.set_model(capi.HostModel(L, capi.host_params("qshmm"), model_path("QSHMM-RSII.model")))
            pe.set_synthetic_sequence(30000000, 1, 7)
            fastq, _, _, _ = pe.simulate(int(20.0 * 30000000), rng_mode=capi.RNG_PHILOX, seed=11)
            pe.close()
            self.pool, _ = capi.sample_filter(L, fastq)
        self.hm = capi.HostModel(L, capi.host_params(wl["method"], **wl["params"]),
                                 model_path(wl["model"]) if wl["model"] else None)
        self.local, self.simulator = local, simulator
        self.options = []
        if overrides:
            for opt, val in (("target_batch_bases", args.batch_bases), ("chain_chunk", args.chain_chunk),
                             ("first_batch_div", args.first_batch_div), ("host_batch_bases", args.host_batch_bases)):
                if val:
                    self.options.append((opt, int(val)))
            if args.bam:
                self.options.append(("bam", 1))
                wl["name"] += " [BAM records]"
        if wl.get("batch_bases") and not (overrides and args.batch_bases):
            self.options.append(("target_batch_bases", int(wl["batch_bases"])))
        self.engines = []
        self.eng = eng = self.engine(0)
        self.depth = wl["depth"]
        self.contigs = [max(200000, int(m * 1000000 * args.scale)) for m in CONTIG_MBP]
        self.bias = [0.0] + [1.0] * 10 + [0.0]
        self.seqset = None
        if wl.get("strategy") == "trans":
            # SURVEY.md 8d C4: log-normal lengths (median 1.5 kb, capped), Zipf expression counts, both strands
            rng = np.random.default_rng(GENOME_SEED)
            nt = max(100, int(wl["n_transcripts"] * args.scale))
            lens = np.clip(np.exp(rng.normal(np.log(1500.0), 0.75, nt)).astype(np.int64), 200, 100000)
            w = 1.0 / np.arange(1, nt + 1) ** 0.9
            expr = rng.permutation(np.maximum(1, (w / w.sum() * wl["n_reads"] * args.scale)).astype(np.int64))
            text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, int(lens.sum()))].tobytes()
            st0 = np.zeros(nt + 1, dtype=np.int64)
            st0[1:] = np.cumsum(lens)
            plus = (expr + 1) // 2
            names = [b"T%06d" % (t + 1) for t in range(nt)]
            id_start = np.zeros(nt + 1, dtype=np.int32)
            id_start[1:] = np.cumsum([len(x) for x in names])
            self.seqset = dict(n=nt, bases=text, start=st0, plus=plus.astype(np.int32),
                               minus=(expr - plus).astype(np.int32), ids=b"".join(names), id_start=id_start)
            self.contigs = [int(lens.sum())]
            self.total_reads = int(expr.sum())
            eng.set_seqset("trans", self.seqset, self.bias)

    def engine(self, lane):
        """engine number `lane` of this GPU (the host-delivery arm drives two, see run_parts)"""
        while len(self.engines) <= lane:
            e = self.simulator.Engine(self.local)
            e.set_model(self.hm)
            for opt, val in self.options:
                e.set_option(opt, val)
            if self.pool is not None:
                e.set_pool(self.pool)
            if self.engines and getattr(self, "seqset", None) is not None:
                e.set_seqset("trans", self.seqset, self.bias)
            self.engines.append(e)
        return self.engines[lane]

    def close(self):
        for e in self.engines:
            e.close()
        self.engines = []

    def run_part(self, part, rng_seed=0, read_range=None, prefix=0, host_seq=None, sink=None, on_chunk=None, eng=None):
        """one part of the run: WGS — a sequence, or a read range of one (part = dict(seq, first_read, max_reads, last),
        stats_reduce.plan_line_split; prefix = emitted bases of the sequence's earlier parts when this is its dependent
        last part); sequence sets — the whole table or this rank's read-number range of it.
        host_seq = None: the sequence text is generated in HBM and the records stay there (device arm);
        otherwise the text is uploaded from that pinned host buffer and every record byte is delivered to host memory.
        Returns (bases, record bytes, stats)."""
        eng, capi = eng or self.eng, self.capi
        device = host_seq is None
        if self.seqset is None:
            k = part["seq"]
            if device:
                eng.set_synthetic_sequence(self.contigs[k], k + 1, GENOME_SEED + k)
            else:
                eng.set_sequence_ptr(host_seq.data_ptr(), self.contigs[k], k + 1, self.bias)
            eng.begin(int(self.depth * self.contigs[k]), rng_mode=capi.RNG_PHILOX, seed=0,
                      first_read=part["first_read"], max_reads=part["max_reads"], len_total_start=prefix)
        else:
            if not device:
                eng.set_seqset("trans", self.seqset, self.bias)  # the table's text goes up with every step
            fr, mr = read_range if read_range else (0, 0)
            eng.begin(0, rng_mode=capi.RNG_PHILOX, seed=1 + rng_seed, first_read=fr, max_reads=mr)
        bases = out_bytes = 0
        while True:
            c = eng.next_chunk(device=device)
            if c is None:
                break
            bases += c.bases
            out_bytes += c.reads_bytes + c.maf_bytes
            if sink is not None and c.reads_bytes:  # the consumer looks at the delivered bytes
                sink[0] ^= C.c_ubyte.from_address(c.reads + c.reads_bytes - 1).value
            if on_chunk is not None:
                on_chunk(c)
        st = eng.end()
        if self.seqset is None and not part["last"]:
            if st.res_num != part["max_reads"] or st.len_total_end >= int(self.depth * self.contigs[part["seq"]]):
                raise RuntimeError("line split: a part that is not the last one of sequence %d reached the quota "
                                   "(the read-count estimate was off by more than the snap margin)" % (part["seq"] + 1))
        return bases, out_bytes, st

    def pilot_mean_emitted(self, k, n_reads=16384):
        """emitted bases per read, from the first n_reads reads of sequence k (a few ms): what the line split needs to
        turn a quota into an estimated read count.  Reads depend only on (seed, sequence, read number), so every rank
        gets the same number without talking to the others."""
        b, _, st = self.run_part(dict(seq=k, first_read=0, max_reads=n_reads, last=True))
        return st.len_total_end / max(1, st.res_num)


def whole_parts(step_ids):
    return [dict(seq=k, first_read=0, max_reads=0, last=True, est=0.0) for k in step_ids]


def run_parts(W, parts, dist, device, on_part, read_range=None, host_seq=None, sink=None, on_chunk=None, lanes=1):
    """this rank's parts in the order of stats_reduce.split_order: feeders, publish (asynchronous all-reduce of the
    emitted bases per sequence), whole sequences, dependent last parts (each told its len_total_start).
    lanes = 2: two engines on this GPU, each driven by its own host thread, take the parts of a PHASE alternately — in
    the host-delivery arm one run's start-up (the next sequence ingested, its first batch generated: nothing to copy for
    15-20 ms) hides behind the other engine's copies; in the device arm kernels bound by different things overlap.
    The phases stay separate on purpose.  Measured on 8 B200 (value of the c3 run): phases 823.7 Gbp/s; one queue over all
    three phases 490 (a feeder that shares its GPU with a whole sequence takes twice as long, and every rank that starts
    with a dependent part waits for the slowest feeder anywhere); feeders alone, then one queue of whole sequences and
    dependent parts 629 (the dependent part is picked up at once and waits for the all-reduce while it could have run
    behind the whole sequences)."""
    from pbsim_b200 import stats_reduce as SR
    feeders, whole, dependent = SR.split_order(parts)
    ex = None
    if W.seqset is None and dist is not None:
        import torch
        ex = SR.SplitExchange(len(W.contigs), dist, device="cuda" if torch.cuda.is_available() else "cpu")
    lock = threading.Lock()
    base = 0
    for phase, plist in (("feed", feeders), ("whole", whole), ("dep", dependent)):
        if phase == "whole" and ex is not None:
            ex.publish()
        nxt = [0]
        errors = []

        def worker(lane):
            try:
                import torch
                if torch.cuda.is_available():
                    torch.cuda.set_device(W.local)  # the current device is a per-thread setting
                while True:
                    with lock:
                        j = nxt[0]
                        nxt[0] += 1
                    if j >= len(plist) or errors:
                        return
                    p = plist[j]
                    prefix = ex.prefix(p["seq"]) if phase == "dep" else 0
                    if on_chunk is not None:
                        on_chunk(p)  # a new part begins
                    b, ob, st = W.run_part(p, rng_seed=(base + j if W.seqset is not None else 0), read_range=read_range,
                                           prefix=prefix, host_seq=None if host_seq is None else host_seq[p["seq"]],
                                           sink=sink, on_chunk=on_chunk, eng=W.engine(lane))
                    with lock:
                        if phase == "feed":
                            ex.add(p["seq"], st.len_total_end)
                        on_part(p, b, ob, st)
            except Exception as ex_:  # noqa: BLE001 - re-raised on the calling thread
                errors.append(ex_)

        n_lanes = min(lanes, len(plist)) if on_chunk is None else 1
        if n_lanes <= 1:
            worker(0)
        else:
            for lane in range(n_lanes):
                W.engine(lane)  # created on this thread, before the clocks of the workers start
            ts = [threading.Thread(target=worker, args=(lane,)) for lane in range(n_lanes)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        if errors:
            raise errors[0]
        base += len(plist)


def measure(W, my_parts, warm_parts, e2e_steps, barrier, dist=None, read_range=None, gzip_arm=True, text_arm=True,
            e2e_warm=False, e2e_lanes=2, parts_e=None, dev_lanes=1):
    """device-resident arm + end-to-end arm(s) over this rank's parts.  Returns a dict of local measurements."""
    import torch
    eng, capi = W.eng, W.capi
    for p in warm_parts:  # warm-up (also grows every arena to its steady-state size)
        W.run_part(dict(p, first_read=0, last=True, max_reads=p["max_reads"]), read_range=read_range)
    dev_lanes = min(dev_lanes, max(1, len(my_parts)))
    for lane in range(1, dev_lanes):  # every engine of the device arm warmed on this rank's largest part
        for p in warm_parts[:1]:
            W.run_part(dict(p, first_read=0, last=True, max_reads=p["max_reads"]), read_range=read_range, eng=W.engine(lane))
    barrier()
    for lane in range(dev_lanes):
        W.engine(lane).timer_start()
    t0 = time.perf_counter()
    acc = dict(bases=0, out_bytes=0, launches=0, sim=0.0, emit=0.0, seg=0.0, chain=0.0, gen=0.0, done=[])

    tp = [time.perf_counter()]

    def on_part(p, b, ob, st):
        if os.environ.get("PBSIM_BENCH_DEBUG"):
            t = time.perf_counter()
            sys.stderr.write("[bench] rank %d part seq %d first_read %d max_reads %d last %s: %.3f Gbase, %.2f ms wall, "
                             "%.2f ms generation\n" % (W.rank, p["seq"] + 1, p["first_read"], p["max_reads"], p["last"],
                                                       b / 1e9, (t - tp[0]) * 1e3, st.gen_seconds * 1e3))
            tp[0] = t
        acc["bases"] += b
        acc["out_bytes"] += ob
        acc["launches"] += st.kernel_launches
        acc["sim"] += st.sim_seconds
        acc["emit"] += st.emit_seconds
        acc["seg"] += st.seg_seconds
        acc["chain"] += st.chain_seconds
        acc["gen"] += st.gen_seconds
        acc["done"].append((p, st))

    run_parts(W, my_parts, dist, True, on_part, read_range=read_range, lanes=dev_lanes)
    # CUDA events on every engine's own stream, all started behind the same device-wide synchronisation: the span of
    # the timed steps is the longest of them
    acc["dev_ms"] = max(W.engine(lane).timer_stop() for lane in range(dev_lanes)) if my_parts else 0.0
    barrier()
    acc["wall_ms"] = (time.perf_counter() - t0) * 1e3
    acc["kern"] = None
    whole_mine = [p for p in my_parts if p["last"] and p["first_read"] == 0]
    if dev_lanes > 1 and whole_mine:
        # kernels of different engines overlap in the timed steps, so their own CUDA-event times there are times under
        # sharing: the per-kernel roofline numbers come from a short single-engine pass (untimed for `value`)
        k1 = dict(bases=0, sim=0.0, emit=0.0, seg=0.0, chain=0.0, gen=0.0, steps=0)
        eng.timer_start()
        for p in whole_mine[:3]:
            b, ob, st = W.run_part(p, read_range=read_range)
            k1["bases"] += b
            k1["steps"] += 1
            for a_, f_ in (("sim", "sim_seconds"), ("emit", "emit_seconds"), ("seg", "seg_seconds"),
                           ("chain", "chain_seconds"), ("gen", "gen_seconds")):
                k1[a_] += getattr(st, f_)
        k1["dev_ms"] = eng.timer_stop()
        acc["kern"] = k1
    acc["e2e"] = acc["e2e_gz"] = None
    # the host-buffer arm runs the same parts (a prefix of the run's sequences when --e2e-steps asks for fewer)
    if parts_e is not None:
        pass  # the caller's plan for the host-delivery arm (pieces proportional to every rank's delivery rate)
    elif e2e_steps >= 0 and W.seqset is None:
        keep = set(sorted(set(p["seq"] for p in my_parts), key=lambda k: [q["seq"] for q in my_parts].index(k))[:e2e_steps])
        parts_e = [p for p in my_parts if p["seq"] in keep] if dist is None else my_parts
    else:
        parts_e = my_parts[:e2e_steps] if e2e_steps >= 0 else my_parts
    if e2e_steps != 0:
        host_seq = {}
        if W.seqset is None:
            for k in sorted(set(p["seq"] for p in parts_e)):  # pinned host copies of the sequence text (untimed preparation)
                eng.set_synthetic_sequence(W.contigs[k], k + 1, GENOME_SEED + k)
                t = torch.empty(W.contigs[k], dtype=torch.uint8, pin_memory=True)
                eng.get_sequence_ascii(t.data_ptr(), W.contigs[k])
                host_seq[k] = t
        else:
            host_seq[0] = True
            parts_e = [dict(p, seq=0) for p in parts_e]

        def e2e_pass():
            barrier()
            t0 = time.perf_counter()
            e = dict(bases=0, h2d=0, d2h=0, gen_s=0.0, gz_s=0.0)
            sink = [0]

            def on_e(p, b, ob, st):
                e["bases"] += b
                e["d2h"] += ob
                e["h2d"] += W.contigs[p["seq"]]
                e["gen_s"] += st.gen_seconds
                e["gz_s"] += st.deflate_seconds

            run_parts(W, parts_e, dist, False, on_e, read_range=read_range, host_seq=host_seq, sink=sink, lanes=e2e_lanes)
            barrier()
            # a step is one run of a sequence (or of the set): exactly one of its parts is the last one
            return dict(e, ms=(time.perf_counter() - t0) * 1e3, steps=sum(1 for p in parts_e if p["last"]))

        # untimed: one run through every engine of the arm, so that pinned staging buffers and record buffers exist
        if parts_e:
            big = max(parts_e, key=lambda p: p.get("est", 0.0))
            for lane in range(e2e_lanes if len(parts_e) > 1 else 1):
                W.run_part(dict(big, first_read=0, last=True), read_range=read_range, host_seq=host_seq[big["seq"]],
                           eng=W.engine(lane))
        if text_arm:
            if e2e_warm:  # untimed pass: every buffer reaches its steady-state size
                e2e_pass()
            acc["e2e"] = e2e_pass()
        if gzip_arm:
            # the records gzip-compressed on the GPU before they cross PCIe (the reference's outputs are .gz files,
            # pbsim.cpp:708-730)
            for e_ in W.engines:
                e_.set_option("deflate", 1)
            if e2e_warm:
                e2e_pass()
            acc["e2e_gz"] = e2e_pass()
            for e_ in W.engines:
                e_.set_option("deflate", 0)
        del host_seq
    return acc


def verify_split(W, my_parts, dist, rank):
    """the parts of every sequence shared by several ranks, delivered as text to host memory, against the same sequence
    simulated whole by rank 0: CRC-32 and byte count of every part's FASTQ and MAF bytes must equal those of the whole
    run's bytes cut at the parts' byte counts.  Untimed; meant for a reduced --scale."""
    import zlib
    import torch
    eng = W.eng
    allparts = [None] * dist.get_world_size()
    dist.all_gather_object(allparts, [dict(p) for p in my_parts])
    nparts = {}
    for plist in allparts:
        for p in plist:
            nparts[p["seq"]] = nparts.get(p["seq"], 0) + 1
    shared = sorted(k for k, n in nparts.items() if n > 1)
    host_seq = {}
    for k in shared:
        eng.set_synthetic_sequence(W.contigs[k], k + 1, GENOME_SEED + k)
        t = torch.empty(W.contigs[k], dtype=torch.uint8, pin_memory=True)
        eng.get_sequence_ascii(t.data_ptr(), W.contigs[k])
        host_seq[k] = t
    recs = []
    cur = [None]

    def on_chunk(c):
        if isinstance(c, dict):  # a new part
            cur[0] = dict(seq=c["seq"], first_read=c["first_read"], fq_len=0, fq_crc=0, maf_len=0, maf_crc=0)
            recs.append(cur[0])
            return
        r = cur[0]
        if c.reads_bytes:
            r["fq_crc"] = zlib.crc32((C.c_char * c.reads_bytes).from_address(c.reads), r["fq_crc"])
            r["fq_len"] += c.reads_bytes
        if c.maf_bytes:
            r["maf_crc"] = zlib.crc32((C.c_char * c.maf_bytes).from_address(c.maf), r["maf_crc"])
            r["maf_len"] += c.maf_bytes

    mine = [p for p in my_parts if p["seq"] in shared]
    run_parts(W, mine, dist, False, lambda *a: None, host_seq=host_seq, on_chunk=on_chunk)
    allrecs = [None] * dist.get_world_size()
    dist.all_gather_object(allrecs, recs)
    out = None
    if rank == 0:
        ok, checked, nbytes = True, 0, 0
        for k in shared:
            parts = sorted((r for rl in allrecs for r in rl if r["seq"] == k), key=lambda r: r["first_read"])
            # the whole sequence, streamed; the running CRCs restart at every part boundary
            state = dict(fq_i=0, maf_i=0, got=[dict(fq_crc=0, maf_crc=0, fq_len=0, maf_len=0) for _ in parts])

            def feed(ptr, n, which):  # every stream (FASTQ, MAF) walks the part list on its own
                off = 0
                key_i = which + "_i"
                while n > 0:
                    i = state[key_i]
                    if i >= len(parts):
                        state["overflow"] = True
                        return
                    room = parts[i][which + "_len"] - state["got"][i][which + "_len"]
                    if room == 0:
                        state[key_i] = i + 1
                        continue
                    take = min(room, n)
                    g = state["got"][i]
                    g[which + "_crc"] = zlib.crc32((C.c_char * take).from_address(ptr + off), g[which + "_crc"])
                    g[which + "_len"] += take
                    off += take
                    n -= take

            def on_whole(c):
                if isinstance(c, dict):
                    return
                if c.reads_bytes:
                    feed(c.reads, c.reads_bytes, "fq")
                if c.maf_bytes:
                    feed(c.maf, c.maf_bytes, "maf")

            W.run_part(dict(seq=k, first_read=0, max_reads=0, last=True), host_seq=host_seq[k], on_chunk=on_whole)
            for pr, g in zip(parts, state["got"]):
                checked += 1
                nbytes += g["fq_len"] + g["maf_len"]
                if (pr["fq_len"], pr["fq_crc"], pr["maf_len"], pr["maf_crc"]) != (g["fq_len"], g["fq_crc"], g["maf_len"], g["maf_crc"]):
                    ok = False
            if state.get("overflow"):
                ok = False
        out = {"ok": ok, "shared_sequences": len(shared), "parts_checked": checked, "bytes_compared": nbytes,
               "how": "CRC-32 + length of every part's FASTQ and MAF bytes == the 1-GPU run's bytes cut at the same offsets"}
    dist.barrier()
    return out


# --dump-outputs: per record stream (FASTQ or SAM, MAF) its first DUMP_HEAD bytes and DUMP_SAMPLE bytes at seeded
# positions over the whole stream (a c3 step writes tens of GB); with the statistics the files take 32 MiB
DUMP_HEAD = 2 << 20
DUMP_SAMPLE = 2 << 20
DUMP_SEED = 20240502
DUMP_STATS = ("res_num", "res_pass_num", "res_len_total", "res_len_min", "res_len_max", "res_sub_num", "res_ins_num",
              "res_del_num", "accuracy_total", "res_len_mean", "res_len_sd", "res_accuracy_mean", "res_accuracy_sd",
              "len_total_end")


class _HbmBytes:
    """n bytes of device memory at ptr, for torch.as_tensor (CUDA array interface, no copy)"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "strides": None,
                                         "version": 2}


class StreamSample:
    """the first `head` bytes of a byte stream that arrives in pieces, and its bytes at the sorted positions `pos`"""

    def __init__(self, pos, head):
        self.pos, self.head_n, self.off, self.head, self.sample = pos, head, 0, [], []

    def feed(self, t):
        """t: the next piece, a 1-D uint8 tensor on any device"""
        import numpy as np
        import torch
        n = t.numel()
        if self.off < self.head_n:
            self.head.append(t[:self.head_n - self.off].cpu())
        lo, hi = np.searchsorted(self.pos, [self.off, self.off + n])
        if hi > lo:
            self.sample.append(t[torch.from_numpy(self.pos[lo:hi] - self.off).to(t.device)].cpu())
        self.off += n

    def arrays(self):
        """(head, sample), one float32 per byte"""
        import numpy as np
        import torch
        return [(torch.cat(x).numpy() if x else np.zeros(0, np.uint8)).astype(np.float32) for x in (self.head, self.sample)]


def dump_outputs(W, parts, done, read_range, out_dir):
    """What the last timed step computed, as .npy files in out_dir: for reads (FASTQ or SAM records) and maf,
    <stream>_head.npy (the first DUMP_HEAD bytes) and <stream>_sample.npy (the bytes at DUMP_SAMPLE positions drawn
    with DUMP_SEED over the stream's length), each byte as a float32; stats.npy (float64) = DUMP_STATS, emitted bases,
    reads bytes, maf bytes.  Every batch of the device arm overwrites the records of the previous one, so the step
    runs again, untimed, on the same engine: once to learn the streams' lengths, once to copy the bytes out.  A read
    depends only on seed, sequence and read number; both runs must end with the timed step's statistics.
    Returns what the JSON line reports: the directory, the step's sequence (a sequence set counts as sequence 1), its
    length and the number of batches its records came in."""
    import numpy as np
    import torch
    from pbsim_b200 import stats_reduce as SR
    order = [p for phase in SR.split_order(parts) for p in phase]
    last = order[-1]
    want = [float(getattr(st, f)) for p, st in done if p is last for f in DUMP_STATS]

    def rerun(on_chunk):
        # rng_seed: run_parts seeds the runs of a sequence set by their place in the order
        b, _, st = W.run_part(last, rng_seed=len(order) - 1, read_range=read_range, on_chunk=on_chunk)
        got = [float(getattr(st, f)) for f in DUMP_STATS]
        if got != want:
            raise RuntimeError("--dump-outputs: the untimed run of the last step differs from the timed one: %s != %s"
                               % (dict(zip(DUMP_STATS, got)), dict(zip(DUMP_STATS, want))))
        return b

    totals = [0, 0, 0]  # reads bytes, maf bytes, batches

    def count(c):
        totals[0] += c.reads_bytes
        totals[1] += c.maf_bytes
        totals[2] += 1

    rerun(count)
    rng = np.random.default_rng(DUMP_SEED)
    streams = [StreamSample(np.unique(rng.integers(0, max(1, n), DUMP_SAMPLE)), DUMP_HEAD) for n in totals[:2]]

    def gather(c):
        torch.cuda.synchronize()  # the engine's kernels run on its own streams
        for s, ptr, n in zip(streams, (c.reads, c.maf), (c.reads_bytes, c.maf_bytes)):
            if n:
                s.feed(torch.as_tensor(_HbmBytes(ptr, n)))

    bases = rerun(gather)
    os.makedirs(out_dir, exist_ok=True)
    for name, s in zip(("reads", "maf"), streams):
        for kind, a in zip(("head", "sample"), s.arrays()):
            np.save(os.path.join(out_dir, "%s_%s.npy" % (name, kind)), a)
    np.save(os.path.join(out_dir, "stats.npy"), np.array(want + [bases] + totals[:2], dtype=np.float64))
    return {"dir": out_dir, "sequence": last["seq"] + 1, "sequence_bp": W.contigs[last["seq"]], "batches": totals[2]}


def roofline_block(method, acc, peak, peak_src):
    """whole-step fraction on top; per-kernel fractions (each kernel against its OWN algorithmic bytes) below"""
    bases = acc["bases"]
    dev_s = acc["dev_ms"] * 1e-3
    achieved = ALGO_BYTES_PER_BASE * bases / dev_s / 1e9 if dev_s > 0 else 0.0
    whole = acc
    kern_note = "CUDA-event times of the kernels inside the timed steps"
    if acc.get("kern"):
        acc = acc["kern"]
        bases, dev_s = acc["bases"], acc["dev_ms"] * 1e-3
        kern_note = ("single-engine pass of %d steps after the timed region (in the timed steps two engines share the "
                     "GPU and their kernels overlap)" % acc["steps"])
    qs_events = method in ("qshmm", "sample")   # 2-byte events per read position
    chain_name = "k_chain_chunk" if qs_events else "k_chain_chunk_err"
    seg_name = "k_sim_seg" if qs_events else "k_sim_seg_err"
    kern = {}
    for name, key, secs in ((chain_name, "k_chain_chunk", acc["chain"]), (seg_name, "k_sim_seg", acc["seg"]),
                            ("k_tile_desc + k_emit_rows + k_emit (pass 2)", "k_emit_rows", acc["emit"])):
        if secs <= 0:   # --method sample has no chain
            continue
        ab = KERNEL_ALGO_BYTES[key] if qs_events or key == "k_emit_rows" else KERNEL_ALGO_BYTES[key] / 2.0
        if method == "sample" and key == "k_sim_seg":
            ab = 3.0    # reads a quality byte of the pool entry, writes the 2-byte event
        a = ab * bases / secs / 1e9 if secs > 0 else 0.0
        ncu = NCU_DRAM_BYTES[key] if method == "qshmm" else None
        kern[name] = {"seconds": secs, "algorithmic_bytes_per_base": ab, "achieved": a, "frac": a / peak if peak else None,
                      "share_of_step": secs / dev_s if dev_s else None,
                      "traffic": ncu["bytes"] if ncu else None,
                      "traffic_per_base": ncu["bytes"] / ncu["positions"] if ncu else None,
                      "traffic_source": (ncu["src"] + ": dram__bytes_read.sum + dram__bytes_write.sum of one launch")
                      if ncu else None}
    dom = max(kern, key=lambda n: kern[n]["seconds"])
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
            "what": "whole step: %.2f algorithmic bytes per emitted base x bases / device time of the timed steps"
                    % ALGO_BYTES_PER_BASE,
            "traffic": kern[dom]["traffic"], "kernel": dom + ", rank 0", "algorithmic_bytes_per_base": ALGO_BYTES_PER_BASE,
            "peak_source": peak_src, "dominant_kernel": dict(kern[dom], name=dom), "kernels": kern,
            "kernels_measured_in": kern_note,
            "kernel_seconds": {"sim": whole["sim"], "emit": whole["emit"], "all_generation": whole["gen"]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink contigs (debugging only; reported in config)")
    ap.add_argument("--e2e-steps", type=int, default=-1, help="steps of the host-buffer arm (default: all)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short runs of the other BASELINE configurations")
    ap.add_argument("--extra-steps", type=int, default=3)
    ap.add_argument("--len-sd", type=float, default=None, help="diagnostics: override --length-sd (0 = equal-length reads)")
    ap.add_argument("--len-mean", type=float, default=None, help="diagnostics: override --length-mean")
    ap.add_argument("--batch-bases", type=float, default=None, help="diagnostics: engine target_batch_bases")
    ap.add_argument("--chain-chunk", type=int, default=None, help="diagnostics: engine chain_chunk (segments per chunk)")
    ap.add_argument("--first-batch-div", type=int, default=None, help="diagnostics: engine first_batch_div")
    ap.add_argument("--host-batch-bases", type=float, default=None, help="diagnostics: engine host_batch_bases")
    ap.add_argument("--bam", action="store_true", help="multi-pass workloads: BAM records / BGZF blocks instead of SAM text")
    ap.add_argument("--part-overhead-gbase", type=float, default=0.45,
                    help="line split: fixed cost of one run in units of emitted Gbase (balances ranks that own many "
                         "short sequences against ranks that own few long ones)")
    ap.add_argument("--lanes", type=int, default=2, choices=[1, 2, 3, 4],
                    help="engines per GPU in the device-resident arm, each driven by its own host thread on alternate parts")
    ap.add_argument("--e2e-lanes", type=int, default=2, choices=[1, 2],
                    help="engines per GPU in the host-delivery arm (2: one run's start-up hides behind the other's copies)")
    ap.add_argument("--no-split", action="store_true",
                    help="N > 1: assign whole sequences to ranks (longest first) instead of cutting the line of reads")
    ap.add_argument("--verify-split", action="store_true",
                    help="N > 1: after the timed runs, rank 0 simulates every shared sequence whole and compares the "
                         "CRC-32 of its bytes, cut at the parts' byte counts, with what the ranks delivered")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU: after the timed steps, write what the last of them computed to DIR as .npy files "
                         "(a seeded sample of its records and its statistics, see dump_outputs), so that two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        raise SystemExit("--dump-outputs needs --impl ours and at least one timed step")
    if args.impl == "reference":
        reference_arm(args, dict(WORKLOADS[args.workload]))
        return

    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs runs on one GPU")
    torch.cuda.set_device(local)
    pin_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        # NCCL's own log (whatever level the caller asked for) goes to stderr: stdout carries the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allsum(x):
        if dist is None:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.item()

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    W = Workload(args.workload, args, local, rank)
    wl = W.wl
    # ---- ONE run split over the ranks (strong scaling).  The timed steps are the sequences (warmup + k) mod 24, k < steps,
    #      each simulated to its own depth quota into its own output files (pbsim.cpp:699-754).  All their reads laid on
    #      one line are cut into `world` pieces of equal estimated work (stats_reduce.plan_line_split): a rank owns whole
    #      sequences plus at most one leading and one trailing read range of a sequence it shares with a neighbour; the
    #      quota cut of a shared sequence needs the emitted bases of its earlier parts: one asynchronous all-reduce.
    #      A sequence set (--strategy trans) is one step and has no quota: split by read-number range.
    read_range = None
    split_info = None
    parts_e = None
    d2h_ceiling, my_d2h = host_d2h_ceiling(barrier, allsum) if args.e2e_steps != 0 else (None, None)
    if W.seqset is None:
        from pbsim_b200 import stats_reduce as SR
        step_ids = [(args.warmup + k) % len(W.contigs) for k in range(args.steps)]
        # (--method sample runs whole sequences: its pool passes make the read numbers depend on the quota)
        if world > 1 and not args.no_split and wl["method"] != "sample":
            mean_emit = W.pilot_mean_emitted(step_ids[0])
            reads_est = [W.depth * W.contigs[k] / mean_emit for k in step_ids]
            # work of a sequence = its bases + a fixed cost per run (ingest, the quota's tail reads, the last partly
            # filled batch: about 4 ms, measured with PBSIM_BENCH_DEBUG=1 on one GPU) expressed in bases
            plan = SR.plan_line_split(reads_est, world,
                                      weights=[W.depth * W.contigs[k] + args.part_overhead_gbase * 1e9 for k in step_ids])
            for r in plan:
                for p in r:
                    p["seq"] = step_ids[p["seq"]]
            mine = plan[rank]
            split_info = {"mean_emitted_bases_per_read": mean_emit,
                          "parts_per_rank": [len(r) for r in plan],
                          "sequences_shared_by_two_ranks": sum(1 for r in plan for p in r if not p["last"])}
            if my_d2h:
                # the host-delivery arm is bound by every rank's device-to-host path, and those differ (on this pool's
                # 8-GPU hosts four GPUs reach 8 GB/s and four 18 GB/s when all copy at once): its pieces are
                # proportional to the rates just measured
                import torch as _t
                rt = _t.tensor([my_d2h], dtype=_t.float64, device="cuda")
                allr = [_t.zeros_like(rt) for _ in range(world)]
                dist.all_gather(allr, rt)
                rates = [float(v[0]) for v in allr]
                plan_e = SR.plan_line_split(reads_est, world, shares=rates,
                                            weights=[W.depth * W.contigs[k] + args.part_overhead_gbase * 1e9 for k in step_ids])
                for r in plan_e:
                    for p in r:
                        p["seq"] = step_ids[p["seq"]]
                parts_e = plan_e[rank]
                split_info["host_delivery_d2h_gb_per_s_per_rank"] = [round(x, 2) for x in rates]
                split_info["host_delivery_parts_per_rank"] = [len(r) for r in plan_e]
        else:
            mine = whole_parts([step_ids[i] for i in lpt_assign([W.contigs[k] for k in step_ids], world)[rank]])
            for p in mine:
                p["est"] = float(W.contigs[p["seq"]])
        warm = [max(mine, key=lambda p: p["est"])] * args.warmup if mine else []
    else:
        from pbsim_b200.stats_reduce import read_range_for_rank
        lo, hi = read_range_for_rank(W.total_reads, rank, world)
        read_range = (lo, hi - lo)
        mine = whole_parts([0] * args.steps)
        warm = whole_parts([0] * args.warmup)
    sampler = ClockSampler(local)
    sampler.start()
    acc = measure(W, mine, warm, args.e2e_steps, barrier, dist=dist, read_range=read_range, e2e_lanes=args.e2e_lanes,
                  parts_e=parts_e, dev_lanes=args.lanes)
    clocks = sampler.stop()
    dumped = dump_outputs(W, mine, acc["done"], read_range, args.dump_outputs) if args.dump_outputs else None

    verified = None
    if args.verify_split and dist is not None and split_info is not None:
        verified = verify_split(W, mine, dist, rank)
    per_rank = None
    if dist is not None:
        import torch as _t
        mine_t = _t.tensor([acc["dev_ms"], acc["bases"] / 1e9, float(len(mine))], dtype=_t.float64, device="cuda")
        allv = [_t.zeros_like(mine_t) for _ in range(world)]
        dist.all_gather(allv, mine_t)
        per_rank = {"dev_ms": [round(float(v[0]), 2) for v in allv], "gbases": [round(float(v[1]), 3) for v in allv],
                    "parts": [int(v[2]) for v in allv]}
    tot_bases = allsum(acc["bases"])
    max_ms = allmax(acc["dev_ms"])
    max_wall = allmax(acc["wall_ms"])
    tot_launches = allsum(acc["launches"])
    e2e_line = {}
    for key in ("e2e", "e2e_gz"):
        if acc[key] is not None or world > 1 and args.e2e_steps != 0:
            e = acc[key] or dict(bases=0, ms=0.0, h2d=0, d2h=0, steps=0, gen_s=0.0, gz_s=0.0)
            e2e_line[key] = dict(bases=allsum(e["bases"]), ms=allmax(e["ms"]), h2d=allsum(e["h2d"]), d2h=allsum(e["d2h"]),
                                 steps=(args.steps if world > 1 else e["steps"]), gen_s=allmax(e["gen_s"]),
                                 gz_s=allmax(e["gz_s"]))
    if dist is not None:
        # the one collective of the path: statistics block (counters + both histograms), NCCL all-reduce
        from pbsim_b200.stats_reduce import allreduce_stats_block
        allreduce_stats_block(W.eng, dist)

    if rank == 0:
        peak, peak_src = measured_peak()
        value = tot_bases / (max_ms * 1e-3) / 1e9 if max_ms > 0 else 0.0
        nsteps = max(1, args.steps)
        config = make_config(wl, args, world)
        line = {
            "metric": "simulated Gbp/s", "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": max_ms / nsteps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": config, "host_wall_ms_per_step": max_wall / nsteps,
            "gpu_launches": int(tot_launches),
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"]},
            "roofline": roofline_block(wl["method"], acc, peak, peak_src),
        }
        if per_rank is not None:
            line["per_rank"] = per_rank
        if dumped is not None:
            line["dump_outputs"] = dumped
        if split_info is not None:
            line["split"] = split_info
            if verified is not None:
                line["split"]["verified"] = verified
        # e2e delivers what the reference's run delivers: gzip-compressed record files (its FASTQ / MAF streams go
        # through `gzip` children into <prefix>_NNNN.fq.gz / .maf.gz, pbsim.cpp:708-730); the engine writes the gzip
        # members on the GPU (option "deflate").  e2e_text is the same run delivering the uncompressed text.
        for key, name, what in (("e2e_gz", "e2e", "gzip members written by the GPU (option deflate): the format of the "
                                                  "reference's output files (.fq.gz / .maf.gz, pbsim.cpp:708-730)"),
                                ("e2e", "e2e_text", "uncompressed text records")):
            if key in e2e_line and e2e_line[key]["ms"] > 0:
                e = e2e_line[key]
                st = max(1.0, e["steps"])
                line[name] = {"value": e["bases"] / (e["ms"] * 1e-3) / 1e9, "unit": "Gbp/s",
                              "h2d_bytes_per_step": e["h2d"] / st, "d2h_bytes_per_step": e["d2h"] / st,
                              "steps": int(e["steps"]), "ms_per_step": e["ms"] / (st / world), "delivered": what,
                              "d2h_gb_per_s": e["d2h"] / (e["ms"] * 1e-3) / 1e9,
                              "device_seconds": {"generation_incl_deflate": e["gen_s"], "of_which_deflate": e["gz_s"],
                                                 "wall": e["ms"] * 1e-3}}
                ceil = d2h_ceiling
                if ceil:
                    line[name]["host_d2h_ceiling_gb_per_s"] = ceil
                    line[name]["d2h_frac_of_host_ceiling"] = line[name]["d2h_gb_per_s"] / ceil
        if "e2e_text" in line and "e2e" in line:
            line["e2e"]["compression_ratio"] = line["e2e_text"]["d2h_bytes_per_step"] / max(1.0, line["e2e"]["d2h_bytes_per_step"])
            line["e2e"]["engines_per_gpu"] = line["e2e_text"]["engines_per_gpu"] = args.e2e_lanes
        # ---- short runs of the other BASELINE configurations (one GPU): value + roofline each
        if world == 1 and not args.no_extras and args.workload == "c3":
            W.close()
            line["extra"] = {}
            for key in ("c1", "c2", "c4", "c5", "cs"):
                try:
                    X = Workload(key, args, local, rank, overrides=False)
                    ns = args.extra_steps if X.seqset is None else 1
                    st_ids = [(2 + k) % len(X.contigs) for k in range(ns)]  # mid-sized contigs
                    xp = whole_parts(st_ids if X.seqset is None else [0] * ns)
                    a = measure(X, xp, xp[:1], 1, barrier, gzip_arm=True, text_arm=False, e2e_warm=True)
                    line["extra"][key] = {
                        "workload": X.wl["name"], "steps": ns,
                        "value": a["bases"] / (a["dev_ms"] * 1e-3) / 1e9, "unit": "Gbp/s",
                        "e2e": a["e2e_gz"]["bases"] / (a["e2e_gz"]["ms"] * 1e-3) / 1e9 if a["e2e_gz"] else None,
                        "roofline": roofline_block(X.wl["method"], a, peak, peak_src)}
                    X.close()
                except Exception as ex:  # an extra must never cost the headline
                    line["extra"][key] = {"error": repr(ex)}
        if not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline(wl)
            except Exception as ex:  # never lose the GPU line to a host-side hiccup
                line["cpu_baseline"] = {"value": None, "unit": "Gbp/s", "cores": 1, "kind": "reference",
                                        "sample": "failed: %r" % (ex,)}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def pin_to_gpu_numa_node(local):
    """host side of the delivery path: run this rank (and allocate its pinned staging buffers) on the NUMA node its
    GPU hangs off, so that 8 ranks do not all stage through node 0"""
    try:
        import torch
        bdf = None
        pr = torch.cuda.get_device_properties(local)
        if hasattr(pr, "pci_bus_id") and hasattr(pr, "pci_device_id"):
            bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        if bdf is None or not os.path.exists("/sys/bus/pci/devices/%s/numa_node" % bdf):
            out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=20).stdout.decode().strip()
            bdf = out[-12:].lower() if len(out) >= 12 else None  # 00000000:1B:00.0 -> 0000:1b:00.0
        if not bdf:
            return None
        node_path = "/sys/bus/pci/devices/%s/numa_node" % bdf
        node = int(open(node_path).read().strip())
        if node < 0:
            return None
        cpus = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        ids = []
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-")
                ids.extend(range(int(a), int(b) + 1))
            elif part:
                ids.append(int(part))
        if ids:
            os.sched_setaffinity(0, ids)
        return node
    except Exception:
        return None


if __name__ == "__main__":
    main()
