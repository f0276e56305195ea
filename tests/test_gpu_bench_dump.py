"""bench.py --dump-outputs.  CPU: the head and the seeded sample of a byte stream that arrives in pieces of any size.
GPU: what the benchmark dumps for its last timed step equals the records and statistics of the same sequence
simulated again through host delivery (a read depends only on seed, sequence and read number)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench as B
from pbsim_b200 import capi, simulator
from tests.golden_util import model_path


@pytest.mark.parametrize("seed", range(6))
def test_stream_sample_is_independent_of_the_pieces(seed):
    rng = np.random.default_rng(seed)
    data = rng.integers(0, 256, int(rng.integers(1, 200000))).astype(np.uint8)
    head = int(rng.choice([1, 1000, 70000, 10 ** 6]))
    pos = np.unique(rng.integers(0, len(data), int(rng.integers(1, 5000))))
    s = B.StreamSample(pos, head)
    cuts = np.unique(np.concatenate([[0, len(data)], rng.integers(0, len(data), int(rng.integers(0, 300)))]))
    for a, b in zip(cuts[:-1], cuts[1:]):  # pieces from 1 byte to the whole stream, many smaller than the head
        s.feed(torch.from_numpy(data[a:b]))
    got_head, got_sample = s.arrays()
    assert got_head.dtype == got_sample.dtype == np.float32
    assert np.array_equal(got_head, data[:head].astype(np.float32))
    assert np.array_equal(got_sample, data[pos].astype(np.float32))


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_last_steps_records(tmp_path):
    # c1 (9 kb reads) with the smallest batches the engine makes (4096 reads): the dumped step's records come in several
    # device batches; 26 steps: more steps than sequences, so sequences repeat
    steps = 26
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(B.ROOT, "bench.py"), "--gpus", "1", "--workload", "c1", "--steps",
                        str(steps), "--warmup", "1", "--scale", "0.2", "--batch-bases", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       timeout=900)
    assert p.returncode == 0, p.stderr.decode()[-3000:]
    line = json.loads(p.stdout.decode().strip().splitlines()[-1])
    assert line["steps"] == line["e2e"]["steps"] == line["e2e_text"]["steps"] == steps
    dumped = line["dump_outputs"]
    assert dumped["dir"] == str(out) and dumped["batches"] > 1
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(got) == ["maf_head", "maf_sample", "reads_head", "reads_sample", "stats"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    k, n = dumped["sequence"] - 1, dumped["sequence_bp"]
    wl = B.WORKLOADS["c1"]
    hm = capi.HostModel(capi.load(), capi.host_params(wl["method"], **wl["params"]), model_path(wl["model"]))
    eng = simulator.Engine(0)
    try:
        eng.set_model(hm)
        eng.set_synthetic_sequence(n, k + 1, B.GENOME_SEED + k)
        reads, maf, st, _ = eng.simulate(int(wl["depth"] * n), rng_mode=capi.RNG_PHILOX, seed=0)
    finally:
        eng.close()
    bases = sum(len(s) for s in reads.split(b"\n")[1::4])  # FASTQ: the sequence is the second line of a record
    want_stats = [float(getattr(st, f)) for f in B.DUMP_STATS] + [bases, len(reads), len(maf)]
    assert got["stats"].tolist() == want_stats
    rng = np.random.default_rng(B.DUMP_SEED)
    for name, text in (("reads", reads), ("maf", maf)):
        b = np.frombuffer(text, dtype=np.uint8)
        assert np.array_equal(got[name + "_head"], b[:B.DUMP_HEAD].astype(np.float32)), name
        pos = np.unique(rng.integers(0, len(b), B.DUMP_SAMPLE))
        assert np.array_equal(got[name + "_sample"], b[pos].astype(np.float32)), name
