"""ctypes declarations of the libpbsim_cuda C ABI (include/pbsim_cuda.h).

This is the thin binding the Python harness (tests/, bench.py) uses; the production host is the
C++ `pbsim` driver (pbsim_b200/csrc/pbsim_main.cpp), which links the same library.
There is no fallback: if the shared library is missing, loading raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpbsim_cuda.so")

NQV = 94
NACC = 101
METHOD_QSHMM = 1
METHOD_ERRHMM = 2
METHOD_SAMPLE = 3
RNG_PHILOX = 0
RNG_REPLAY = 1


class HmmRow(C.Structure):
    _fields_ = [
        ("exists", C.c_int32),
        ("nstates", C.c_int32),
        ("resolution", C.c_int32),
        ("init_mod", C.c_int32),
        ("init", C.POINTER(C.c_uint8)),
        ("tran_mod", C.POINTER(C.c_int32)),
        ("tran", C.POINTER(C.c_uint8)),
        ("emis_mod", C.POINTER(C.c_int32)),
        ("emis", C.POINTER(C.c_uint8)),
        ("emis_del", C.POINTER(C.c_int32)),
        ("freq_mod", C.c_int32),
        ("freq", C.POINTER(C.c_uint8)),
    ]


class Model(C.Structure):
    _fields_ = [
        ("method", C.c_int32),
        ("pass_num", C.c_int32),
        ("len_min", C.c_int64),
        ("len_max", C.c_int64),
        ("accuracy_mean", C.c_double),
        ("id_prefix", C.c_char * 128),
        ("prob2len", C.POINTER(C.c_int32)),
        ("len_rand_value", C.c_int32),
        ("prob2accuracy", C.POINTER(C.c_uint8)),
        ("accuracy_rand_value", C.c_int32),
        ("acc_lo", C.c_int32),
        ("acc_hi", C.c_int32),
        ("sub_thre", C.c_int32 * NQV),
        ("ins_thre", C.c_int32 * NQV),
        ("del_thre", C.c_int32 * NQV),
        ("qc_prob", C.c_double * NQV),
        ("model_acc_min", C.c_int32),
        ("model_acc_max", C.c_int32),
        ("rows", HmmRow * NACC),
    ]


class Sequence(C.Structure):
    _fields_ = [
        ("bases", C.c_char_p),
        ("len", C.c_int64),
        ("seq_num", C.c_int32),
        ("hp_del_bias", C.c_double * 12),
    ]


STRATEGY_WGS, STRATEGY_TRANS, STRATEGY_TEMPL = 0, 1, 2


class SeqSet(C.Structure):
    _fields_ = [
        ("strategy", C.c_int32),
        ("n", C.c_int64),
        ("bases", C.c_void_p),
        ("start", C.c_void_p),
        ("plus_exp", C.c_void_p),
        ("minus_exp", C.c_void_p),
        ("ids", C.c_void_p),
        ("id_start", C.c_void_p),
        ("hp_del_bias", C.c_double * 12),
    ]


class Run(C.Structure):
    _fields_ = [
        ("rng_mode", C.c_int32),
        ("seed", C.c_uint32),
        ("len_quota", C.c_int64),
        ("first_read", C.c_int64),
        ("len_total_start", C.c_int64),
        ("max_reads", C.c_int64),
        ("batch_reads", C.c_int64),
        ("replay_draws", C.c_void_p),
        ("replay_ndraws", C.c_int64),
        ("replay_starts", C.c_void_p),
        ("replay_nsubreads", C.c_int64),
    ]


class Chunk(C.Structure):
    _fields_ = [
        ("reads", C.c_void_p),
        ("reads_bytes", C.c_int64),
        ("maf", C.c_void_p),
        ("maf_bytes", C.c_int64),
        ("first_read", C.c_int64),
        ("n_reads", C.c_int64),
        ("bases", C.c_int64),
        ("on_device", C.c_int32),
        ("compressed", C.c_int32),
        ("reads_text_bytes", C.c_int64),
        ("maf_text_bytes", C.c_int64),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("res_num", C.c_int64),
        ("res_pass_num", C.c_int64),
        ("res_len_total", C.c_int64),
        ("res_len_min", C.c_int64),
        ("res_len_max", C.c_int64),
        ("res_sub_num", C.c_int64),
        ("res_ins_num", C.c_int64),
        ("res_del_num", C.c_int64),
        ("accuracy_total", C.c_double),
        ("res_len_mean", C.c_double),
        ("res_len_sd", C.c_double),
        ("res_accuracy_mean", C.c_double),
        ("res_accuracy_sd", C.c_double),
        ("gen_seconds", C.c_double),
        ("sim_seconds", C.c_double),
        ("emit_seconds", C.c_double),
        ("deflate_seconds", C.c_double),
        ("seg_seconds", C.c_double),
        ("kernel_launches", C.c_int64),
        ("chain_seconds", C.c_double),
        ("len_total_end", C.c_int64),
    ]


class HostParams(C.Structure):
    _fields_ = [
        ("method", C.c_int32),
        ("pass_num", C.c_int32),
        ("len_min", C.c_int64),
        ("len_max", C.c_int64),
        ("len_mean", C.c_double),
        ("len_sd", C.c_double),
        ("accuracy_mean", C.c_double),
        ("sub_ratio", C.c_int64),
        ("ins_ratio", C.c_int64),
        ("del_ratio", C.c_int64),
        ("id_prefix", C.c_char * 128),
    ]


class SampleStats(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("num", "len_total", "len_min", "len_max", "num_filtered", "len_total_filtered",
                                         "len_min_filtered", "len_max_filtered")] + [
        (k, C.c_double) for k in ("len_mean_filtered", "len_sd_filtered", "accuracy_mean_filtered",
                                  "accuracy_sd_filtered")]


HOST_EXPORTS = ["pbsim_host_sample_filter", "pbsim_host_model_load", "pbsim_host_model_get", "pbsim_host_model_free", "pbsim_host_hp_del_bias",
                "pbsim_host_ssp_table", "pbsim_host_deflate_code"]
ENGINE_EXPORTS = [
    "pbsim_cuda_abi_version", "pbsim_cuda_last_error", "pbsim_cuda_create", "pbsim_cuda_destroy",
    "pbsim_cuda_set_model", "pbsim_cuda_set_sequence", "pbsim_cuda_set_seqset", "pbsim_cuda_set_pool", "pbsim_cuda_set_synthetic_sequence",
    "pbsim_cuda_update_hp_del_bias", "pbsim_cuda_get_sequence_ascii", "pbsim_cuda_get_sequence_tables", "pbsim_cuda_get_hpfreq",
    "pbsim_cuda_simulate_begin", "pbsim_cuda_next_chunk",
    "pbsim_cuda_next_chunk_device", "pbsim_cuda_simulate_end", "pbsim_cuda_stats_device_block",
    "pbsim_cuda_last_chunk_info", "pbsim_cuda_device_timer", "pbsim_cuda_set_option",
    "pbsim_cuda_set_sequence_name",
]


def declare_host(L):
    """Prototypes of the host front end (present in libpbsim_cuda.so and in the tests' hostsim build)."""
    L.pbsim_host_model_load.restype = C.c_int
    L.pbsim_host_model_load.argtypes = [C.POINTER(C.c_void_p), C.POINTER(HostParams), C.c_char_p,
                                        C.POINTER(C.c_char_p)]
    L.pbsim_host_model_get.restype = C.POINTER(Model)
    L.pbsim_host_model_get.argtypes = [C.c_void_p]
    L.pbsim_host_model_free.restype = None
    L.pbsim_host_model_free.argtypes = [C.c_void_p]
    L.pbsim_host_hp_del_bias.restype = None
    L.pbsim_host_hp_del_bias.argtypes = [C.c_double, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    L.pbsim_host_deflate_code.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p, C.c_int32]
    L.pbsim_host_sample_filter.argtypes = [C.c_char_p, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_double,
                                           C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                           C.POINTER(SampleStats), C.POINTER(C.c_char_p)]
    L.pbsim_host_ssp_table.restype = None
    L.pbsim_host_ssp_table.argtypes = [C.c_int32, C.c_void_p, C.c_void_p]
    return L


def declare_engine(L):
    L.pbsim_cuda_abi_version.restype = C.c_int
    L.pbsim_cuda_last_error.restype = C.c_char_p
    L.pbsim_cuda_last_error.argtypes = [C.c_void_p]
    L.pbsim_cuda_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.pbsim_cuda_destroy.restype = None
    L.pbsim_cuda_destroy.argtypes = [C.c_void_p]
    L.pbsim_cuda_set_model.argtypes = [C.c_void_p, C.POINTER(Model)]
    L.pbsim_cuda_set_sequence.argtypes = [C.c_void_p, C.POINTER(Sequence)]
    L.pbsim_cuda_set_sequence_name.restype = C.c_int
    L.pbsim_cuda_set_sequence_name.argtypes = [C.c_void_p, C.c_char_p]
    L.pbsim_cuda_set_seqset.argtypes = [C.c_void_p, C.POINTER(SeqSet)]
    L.pbsim_cuda_set_pool.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]
    L.pbsim_cuda_set_synthetic_sequence.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_uint64]
    L.pbsim_cuda_update_hp_del_bias.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.pbsim_cuda_get_sequence_ascii.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    L.pbsim_cuda_get_sequence_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    L.pbsim_cuda_get_hpfreq.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.pbsim_cuda_simulate_begin.argtypes = [C.c_void_p, C.POINTER(Run)]
    L.pbsim_cuda_next_chunk.argtypes = [C.c_void_p, C.POINTER(Chunk)]
    L.pbsim_cuda_next_chunk_device.argtypes = [C.c_void_p, C.POINTER(Chunk)]
    L.pbsim_cuda_simulate_end.argtypes = [C.c_void_p, C.POINTER(Stats), C.c_void_p, C.c_int64, C.c_void_p]
    L.pbsim_cuda_stats_device_block.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    L.pbsim_cuda_device_timer.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    L.pbsim_cuda_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
    L.pbsim_cuda_last_chunk_info.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    return L


_lib = None


def load():
    """Load libpbsim_cuda.so (built in-tree by __graft_entry__.build()).  Fails loudly if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libpbsim_cuda.so is not built (%s): run `python -c 'import __graft_entry__ as g; "
                               "g.build()'`; there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        declare_host(L)
        declare_engine(L)
        _lib = L
    return _lib


def truncate_accuracy(x):
    """set_sim_param truncates accuracy options to two decimals: int(x*100)*0.01 (pbsim.cpp:1620-1660)."""
    return int(x * 100) * 0.01


def host_params(method, pass_num=1, accuracy_mean=0.85, accuracy_mean_set=False, len_min=100, len_max=1000000,
                len_mean=9000.0, len_sd=7000.0, ratio=(6, 55, 39), id_prefix="S", **_ignored):
    p = HostParams()
    p.method = (METHOD_SAMPLE if method in ("sample", METHOD_SAMPLE)
                else METHOD_QSHMM if method in ("qshmm", METHOD_QSHMM) else METHOD_ERRHMM)
    p.pass_num = pass_num
    p.len_min, p.len_max = len_min, len_max
    p.len_mean, p.len_sd = len_mean, len_sd
    p.accuracy_mean = truncate_accuracy(accuracy_mean) if accuracy_mean_set else accuracy_mean
    p.sub_ratio, p.ins_ratio, p.del_ratio = ratio
    p.id_prefix = id_prefix.encode()
    return p


class HostModel:
    """Owns a pbsim_host_model (parsed model + quantised tables)."""

    def __init__(self, L, params, model_path):
        self.L = L
        self.h = C.c_void_p()
        err = C.c_char_p()
        rc = L.pbsim_host_model_load(C.byref(self.h), C.byref(params), model_path.encode() if model_path else None,
                                     C.byref(err))
        if rc != 0:
            raise RuntimeError("pbsim_host_model_load: %s (%d)" % ((err.value or b"").decode(), rc))
        self.params = params

    @property
    def ptr(self):
        return self.L.pbsim_host_model_get(self.h)

    @property
    def view(self):
        return self.ptr.contents

    def close(self):
        if self.h:
            self.L.pbsim_host_model_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def hp_del_bias(L, opt, hpfreq12):
    arr = (C.c_int64 * 12)(*[int(x) for x in hpfreq12])
    out = (C.c_double * 12)()
    L.pbsim_host_hp_del_bias(opt, arr, out)
    return list(out)


def sample_filter(L, fastq, len_min=100, len_max=1000000, accuracy_min=0.75, accuracy_max=1.0):
    """get_sample_inf (pbsim.cpp:1155): -> (pool of quality strings in file order, SampleStats)"""
    import numpy as np
    quals = C.create_string_buffer(max(len(fastq), 1))
    cap = fastq.count(b"\n") // 4 + 2
    qstart = np.zeros(cap, dtype=np.int64)
    n = C.c_int64()
    st = SampleStats()
    err = C.c_char_p()
    rc = L.pbsim_host_sample_filter(fastq, len(fastq), len_min, len_max, accuracy_min, accuracy_max, quals,
                                    qstart.ctypes.data, cap, C.byref(n), C.byref(st), C.byref(err))
    if rc != 0:
        raise RuntimeError((err.value or b"").decode())
    raw = quals.raw
    return [raw[qstart[i]:qstart[i + 1]] for i in range(n.value)], st


def format_sample_stats(st, file_name):
    """print_sample_stats (pbsim.cpp:1336-1358)"""
    return (":::: sample reads stats ::::\n\nfile name : %s\n\n:: all reads ::\nread num. : %d\nread total length : %d\n"
            "read min length : %d\nread max length : %d\n\n:: filtered reads ::\nread num. : %d\nread total length : %d\n"
            "read min length : %d\nread max length : %d\nread length mean (SD) : %f (%f)\n"
            "read accuracy mean (SD) : %f (%f)\n\n"
            % (file_name, st.num, st.len_total, st.len_min, st.len_max, st.num_filtered, st.len_total_filtered,
               st.len_min_filtered, st.len_max_filtered, st.len_mean_filtered, st.len_sd_filtered,
               st.accuracy_mean_filtered, st.accuracy_sd_filtered))
