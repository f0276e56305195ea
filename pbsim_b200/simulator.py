"""Python harness over the libpbsim_cuda C ABI: the WGS flow of the reference's main()
(pbsim.cpp:666-754) expressed as calls into the engine.  Used by tests/ and bench.py; the production
host is the C++ `pbsim` driver.  Every call goes through the C ABI — no computation happens here.
"""
import ctypes as C

import numpy as np

from . import capi


class EngineError(RuntimeError):
    pass


class Engine:
    def __init__(self, device=0):
        self.L = capi.load()
        self.h = C.c_void_p()
        rc = self.L.pbsim_cuda_create(C.byref(self.h), device)
        if rc != 0:
            raise EngineError("pbsim_cuda_create: %s (%d)" % (self.L.pbsim_cuda_last_error(None).decode(), rc))
        self.model = None
        self._keep = []

    def _chk(self, rc, what):
        if rc < 0:
            raise EngineError("%s: %s (%d)" % (what, self.L.pbsim_cuda_last_error(self.h).decode(), rc))
        return rc

    def close(self):
        if self.h:
            self.L.pbsim_cuda_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_model(self, host_model):
        self.model = host_model  # keeps the tables alive
        self._chk(self.L.pbsim_cuda_set_model(self.h, host_model.ptr), "set_model")

    def set_sequence(self, bases, seq_num, bias):
        s = capi.Sequence()
        self._keep = [bases]
        s.bases = bases
        s.len = len(bases)
        s.seq_num = seq_num
        s.hp_del_bias = (C.c_double * 12)(*bias)
        self._chk(self.L.pbsim_cuda_set_sequence(self.h, C.byref(s)), "set_sequence")
        self.glen = len(bases)

    @staticmethod
    def pack_seqset(seqset):
        """[(name, plus, minus, bases)] -> the concatenated arrays pbsim_seqset points to"""
        names = [x[0].encode() if isinstance(x[0], str) else x[0] for x in seqset]
        bases = b"".join(x[3] for x in seqset)
        start = np.zeros(len(seqset) + 1, dtype=np.int64)
        start[1:] = np.cumsum([len(x[3]) for x in seqset])
        plus = np.array([x[1] for x in seqset], dtype=np.int32)
        minus = np.array([x[2] for x in seqset], dtype=np.int32)
        ids = b"".join(names)
        id_start = np.zeros(len(seqset) + 1, dtype=np.int32)
        id_start[1:] = np.cumsum([len(x) for x in names])
        return dict(n=len(seqset), bases=bases, start=start, plus=plus, minus=minus, ids=ids, id_start=id_start)

    def set_sequence_name(self, name):
        """RNAME of the alignment lines (option "align") of the current WGS sequence; set after set_sequence"""
        self._chk(self.L.pbsim_cuda_set_sequence_name(self.h, name.encode() if isinstance(name, str) else name),
                  "set_sequence_name")

    def set_seqset(self, strategy, seqset, bias):
        """strategy 'trans' | 'templ'; seqset = [(name, plus, minus, bases)] as parsed from the transcript table /
        template FASTA (pbsim.cpp:1075, :1366), or the result of pack_seqset"""
        k = seqset if isinstance(seqset, dict) else self.pack_seqset(seqset)
        self._keep = [k]
        s = capi.SeqSet()
        s.strategy = capi.STRATEGY_TRANS if strategy == "trans" else capi.STRATEGY_TEMPL
        s.n = k["n"]
        s.bases = C.cast(C.c_char_p(k["bases"]), C.c_void_p)
        s.start = k["start"].ctypes.data
        s.plus_exp = k["plus"].ctypes.data
        s.minus_exp = k["minus"].ctypes.data
        s.ids = C.cast(C.c_char_p(k["ids"]), C.c_void_p)
        s.id_start = k["id_start"].ctypes.data
        s.hp_del_bias = (C.c_double * 12)(*bias)
        self._chk(self.L.pbsim_cuda_set_seqset(self.h, C.byref(s)), "set_seqset")
        self.glen = len(k["bases"])

    def set_pool(self, pool):
        """--method sample: the quality strings get_sample_inf keeps (pbsim.cpp:1214-1275), in file order"""
        quals = b"".join(pool)
        qstart = np.zeros(len(pool) + 1, dtype=np.int64)
        qstart[1:] = np.cumsum([len(x) for x in pool])
        self._chk(self.L.pbsim_cuda_set_pool(self.h, quals, qstart.ctypes.data, len(pool)), "set_pool")

    def set_synthetic_sequence(self, length, seq_num, seed):
        self._chk(self.L.pbsim_cuda_set_synthetic_sequence(self.h, length, seq_num, seed), "set_synthetic_sequence")
        self.glen = length

    def set_sequence_ptr(self, ptr, length, seq_num, bias):
        """same as set_sequence, from a raw host pointer (e.g. pinned memory)"""
        s = capi.Sequence()
        s.bases = C.cast(ptr, C.c_char_p)
        s.len = length
        s.seq_num = seq_num
        s.hp_del_bias = (C.c_double * 12)(*bias)
        self._chk(self.L.pbsim_cuda_set_sequence(self.h, C.byref(s)), "set_sequence")
        self.glen = length

    def get_sequence_ascii(self, dst_ptr, cap):
        self._chk(self.L.pbsim_cuda_get_sequence_ascii(self.h, dst_ptr, cap), "get_sequence_ascii")

    def update_bias(self, bias):
        self._chk(self.L.pbsim_cuda_update_hp_del_bias(self.h, (C.c_double * 12)(*bias)), "update_hp_del_bias")

    def set_option(self, name, value):
        self._chk(self.L.pbsim_cuda_set_option(self.h, name.encode(), int(value)), "set_option")

    def timer_start(self):
        self._chk(self.L.pbsim_cuda_device_timer(self.h, 0, None), "device_timer")

    def timer_stop(self):
        ms = C.c_double()
        self._chk(self.L.pbsim_cuda_device_timer(self.h, 1, C.byref(ms)), "device_timer")
        return ms.value

    def stats_block(self):
        ptr = C.c_void_p()
        cells = C.c_int64()
        self._chk(self.L.pbsim_cuda_stats_device_block(self.h, C.byref(ptr), C.byref(cells)), "stats_device_block")
        return ptr.value, cells.value

    def hpfreq(self):
        out = (C.c_int64 * 12)()
        self._chk(self.L.pbsim_cuda_get_hpfreq(self.h, out), "get_hpfreq")
        return list(out)

    def begin(self, len_quota, rng_mode=capi.RNG_PHILOX, seed=0, replay_draws=None, replay_starts=None,
              first_read=0, len_total_start=0, max_reads=0, batch_reads=0):
        run = capi.Run()
        run.rng_mode = rng_mode
        run.seed = seed
        run.len_quota = int(len_quota)
        run.first_read = first_read
        run.len_total_start = len_total_start
        run.max_reads = max_reads
        run.batch_reads = batch_reads
        if rng_mode == capi.RNG_REPLAY and replay_draws is not None and replay_starts is not None:
            d = np.ascontiguousarray(replay_draws, dtype=np.int32)
            s = np.ascontiguousarray(replay_starts, dtype=np.int64)
            self._replay_keep = (d, s)
            run.replay_draws = d.ctypes.data
            run.replay_ndraws = d.size
            run.replay_starts = s.ctypes.data
            run.replay_nsubreads = s.size
        self._chk(self.L.pbsim_cuda_simulate_begin(self.h, C.byref(run)), "simulate_begin")

    def next_chunk(self, device=False):
        c = capi.Chunk()
        f = self.L.pbsim_cuda_next_chunk_device if device else self.L.pbsim_cuda_next_chunk
        rc = self._chk(f(self.h, C.byref(c)), "next_chunk")
        return c if rc == 1 else None

    def end(self, want_hist=False):
        st = capi.Stats()
        if want_hist:
            cells = 2 * self.model.view.len_max + 2
            fl = np.zeros(cells, dtype=np.int64)
            fa = np.zeros(100001, dtype=np.int64)
            self._chk(self.L.pbsim_cuda_simulate_end(self.h, C.byref(st), fl.ctypes.data, cells, fa.ctypes.data),
                      "simulate_end")
            return st, fl, fa
        self._chk(self.L.pbsim_cuda_simulate_end(self.h, C.byref(st), None, 0, None), "simulate_end")
        return st

    def last_chunk_info(self):
        n = C.c_int64()
        self._chk(self.L.pbsim_cuda_last_chunk_info(self.h, None, 0, C.byref(n)), "last_chunk_info")
        out = np.zeros((n.value, 8), dtype=np.int64)
        self._chk(self.L.pbsim_cuda_last_chunk_info(self.h, out.ctypes.data, n.value, C.byref(n)), "last_chunk_info")
        return out

    def simulate(self, len_quota, **kw):
        """Run to the quota, collecting host chunks.  Returns (reads_bytes, maf_bytes, stats, n_chunks)."""
        want_hist = kw.pop("want_hist", False)
        self.begin(len_quota, **kw)
        reads, maf, n = [], [], 0
        while True:
            c = self.next_chunk()
            if c is None:
                break
            reads.append(C.string_at(c.reads, c.reads_bytes))
            maf.append(C.string_at(c.maf, c.maf_bytes))
            n += 1
        st = self.end(want_hist)
        return b"".join(reads), b"".join(maf), st, n


def format_stats(st, seq_num, glen, pass_num):
    """print_simulation_stats for WGS (pbsim.cpp:5541-5564)."""
    depth = st.res_len_total / glen / pass_num
    tot = st.res_len_total
    return (
        ":::: Simulation stats (ref.%d) ::::\n\n" % seq_num
        + "read num. : %d\n" % st.res_num
        + "depth : %f\n" % depth
        + "read length mean (SD) : %f (%f)\n" % (st.res_len_mean, st.res_len_sd)
        + "read length min : %d\n" % st.res_len_min
        + "read length max : %d\n" % st.res_len_max
        + "read accuracy mean (SD) : %f (%f)\n" % (st.res_accuracy_mean, st.res_accuracy_sd)
        + "substitution rate. : %f\n" % (st.res_sub_num / tot)
        + "insertion rate. : %f\n" % (st.res_ins_num / tot)
        + "deletion rate. : %f\n" % (st.res_del_num / tot)
        + "\n"
    )


SAM_HEADER = (b"@HD\tVN:1.5\tSO:unknown\tpb:3.0.7\n"
              b"@RG\tID:ffffffff\tPL:PACBIO\tDS:READTYPE=SUBREAD;Ipd:CodecV1=ip;PulseWidth:CodecV1=pw;"
              b"BINDINGKIT=101-789-500;SEQUENCINGKIT=101-826-100;BASECALLERVERSION=5.0.0;FRAMERATEHZ=100.000000"
              b"\tPU:%s%d\tPM:SEQUELII\n")


class WgsRun:
    """main()'s WGS loop (pbsim.cpp:666-754): per sequence ingest -> bias -> simulate -> stats."""

    def __init__(self, engine, host_model, depth, hp_del_bias=1.0):
        self.e = engine
        self.hm = host_model
        self.depth = depth
        self.opt = hp_del_bias
        self.hp11_running = 0  # genome.hpfreq[11], which aliases hp_del_bias[0] in the reference build
        self.base_bias = [0.0] + [1.0] * 10 + [0.0]
        engine.set_model(host_model)

    def prepass(self, contigs):
        """--hp-del-bias != 1: hpfreq over all sequences first (pbsim.cpp:678-697)."""
        tot = [0] * 12
        for i, (_, s) in enumerate(contigs, start=1):
            self.e.set_sequence(s, i, self.base_bias)
            f = self.e.hpfreq()
            for k in range(12):
                tot[k] += f[k]
        self.hp11_running = tot[11]
        self.base_bias = capi.hp_del_bias(self.e.L, self.opt, tot)

    def simulate_sequence(self, bases, seq_num, name=None, **kw):
        """name: RNAME of the alignment lines (option "align")"""
        bias = list(self.base_bias)
        self.e.set_sequence(bases, seq_num, bias)
        if name is not None:
            self.e.set_sequence_name(name)
        f = self.e.hpfreq()
        self.hp11_running += f[11]
        bias[0] = float(np.array([self.hp11_running], dtype=np.int64).view(np.float64)[0])
        self.e.update_bias(bias)
        quota = int(self.depth * len(bases))
        reads, maf, st, n = self.e.simulate(quota, **kw)
        text = format_stats(st, seq_num, len(bases), self.hm.view.pass_num)
        return reads, maf, st, text


def format_stats_set(st):
    """print_simulation_stats for the transcript / template strategies (pbsim.cpp:5547-5564)."""
    tot = st.res_len_total
    return (
        ":::: Simulation stats ::::\n\n"
        + "read num. : %d\n" % st.res_num
        + "read length mean (SD) : %f (%f)\n" % (st.res_len_mean, st.res_len_sd)
        + "read length min : %d\n" % st.res_len_min
        + "read length max : %d\n" % st.res_len_max
        + "read accuracy mean (SD) : %f (%f)\n" % (st.res_accuracy_mean, st.res_accuracy_sd)
        + "substitution rate. : %f\n" % (st.res_sub_num / tot)
        + "insertion rate. : %f\n" % (st.res_ins_num / tot)
        + "deletion rate. : %f\n" % (st.res_del_num / tot)
        + "\n"
    )


class SetRun:
    """main()'s transcript / template branches (pbsim.cpp:760-868): ingest the set, bias, simulate, stats."""

    def __init__(self, engine, host_model, strategy, hp_del_bias=1.0):
        self.e = engine
        self.hm = host_model
        self.strategy = strategy
        self.opt = hp_del_bias
        engine.set_model(host_model)

    def simulate(self, seqset, **kw):
        bias = [0.0] + [1.0] * 10 + [0.0]
        self.e.set_seqset(self.strategy, seqset, bias)
        if self.opt != 1.0:
            # the --hp-del-bias prepass (:2671-2746, :3244-3310): expression-weighted homopolymer histogram; its
            # cell [11] lands on hp_del_bias[0] in the reference build
            bias = capi.hp_del_bias(self.e.L, self.opt, self.e.hpfreq())
            self.e.set_seqset(self.strategy, seqset, bias)
        reads, maf, st, n = self.e.simulate(0, **kw)
        return reads, maf, st, format_stats_set(st)
