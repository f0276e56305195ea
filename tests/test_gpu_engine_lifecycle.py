"""-m gpu: what an engine leaves behind.  Destroying an engine returns all its device memory, and engines on different
devices of one process each set up the kernels they launch."""
import gzip
import statistics

import pytest
import torch

from pbsim_b200 import capi, simulator
from tests.golden_util import model_path

pytestmark = pytest.mark.gpu


def test_destroy_returns_the_pool():
    """--method sample keeps its quality pool in HBM: six engines with a 256 MB pool each must not use up memory"""
    pool = [b"I" * 1000000] * 256
    free = [torch.cuda.mem_get_info()[0]]
    for _ in range(6):
        eng = simulator.Engine(0)
        eng.set_pool(pool)
        eng.close()
        free.append(torch.cuda.mem_get_info()[0])
    drops = [a - b for a, b in zip(free, free[1:])]
    # the median: other work on the GPU can move the free memory of a single cycle
    assert statistics.median(drops) < 64 << 20, drops


def _deflated_run(device):
    """test_gpu_gzip.py::test_many_batches_and_small_pieces on one device: plain text, then gzip members"""
    eng = simulator.Engine(device)
    try:
        eng.set_model(capi.HostModel(capi.load(), capi.host_params("qshmm"), model_path("QSHMM-RSII.model")))
        n = 1000000
        eng.set_synthetic_sequence(n, 1, 5)
        ref = eng.simulate(2 * n, rng_mode=capi.RNG_PHILOX, seed=9)
        eng.set_option("deflate", 1)
        eng.set_option("stage_bytes", 4096)
        got = eng.simulate(2 * n, rng_mode=capi.RNG_PHILOX, seed=9, batch_reads=37)
    finally:
        eng.close()
    assert got[3] > 50
    assert gzip.decompress(got[0]) == ref[0]
    assert gzip.decompress(got[1]) == ref[1]
    return ref, got


def test_engines_on_two_devices_in_one_process():
    """k_gz_encode needs more dynamic shared memory than a launch gets by default; the attribute that grants it is
    set per device, so the engine on the second device must set it as well"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ref0, got0 = _deflated_run(0)
    ref1, got1 = _deflated_run(1)
    assert ref1[:2] == ref0[:2]
    assert gzip.decompress(got1[0]) == ref0[0]
    assert gzip.decompress(got1[1]) == ref0[1]
    for st in (got0[2], ref1[2], got1[2]):
        for f in ("res_num", "res_len_total", "res_len_min", "res_len_max", "res_sub_num", "res_ins_num", "res_del_num",
                  "accuracy_total"):
            assert getattr(st, f) == getattr(ref0[2], f), f
