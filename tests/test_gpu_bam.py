"""-m gpu: BAM output (option "bam").  With --pass-num > 1 the reference pipes SAM text into `samtools view -b`
(pbsim.cpp:715-722); samtools is not in the image, so the engine's BAM records are decoded by the independent
reader in tests/bam_util.py and compared with the reference's SAM text (golden, replay mode) byte for byte."""
import numpy as np
import pytest

from oracle import oracle as O
from pbsim_b200 import capi, simulator
from tests import bam_util as B
from tests.golden_util import Case, SetCase
from tests.gpu_util import run_case_on_gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = simulator.Engine(0)
    yield e
    e.set_option("bam", 0)
    e.set_option("deflate", 0)
    e.close()


@pytest.mark.parametrize("name", ["err_sequel_multipass", "qs_rsii_multipass"])
@pytest.mark.parametrize("deflate", [0, 1])
def test_bam_records_decode_to_the_reference_sam(eng, name, deflate):
    c = Case(name)
    out, _ = c.run_oracle("glibc")
    eng.set_option("bam", 1)
    eng.set_option("deflate", deflate)
    try:
        res = run_case_on_gpu(c, eng, "replay", oracle_out=out)
    finally:
        eng.set_option("bam", 0)
        eng.set_option("deflate", 0)
    for i, (reads, maf, st, text) in enumerate(res, start=1):
        raw = b"".join(pl for _, pl in B.bgzf_blocks(reads)) if deflate else reads
        assert B.records_to_sam(raw) == c.reads(i), "BAM records differ from the reference's SAM lines, seq %d" % i
        assert text == c.stats_blocks[i]


def test_bam_of_a_template_run_with_odd_lengths_and_lower_case(eng):
    """templates: whole-sequence reads of every length parity, lower-case first bases (nibble N... no: 'a' -> A)"""
    c = SetCase("tm_err_sequel_multipass")
    draws = O.glibc_rand(c.seed, c.ndraws)
    starts = np.concatenate([[0], c.marks[:-1]]).astype(np.int64)
    hm = capi.HostModel(capi.load(), capi.host_params(c.method, **c.okw), c.model)
    run = simulator.SetRun(eng, hm, c.strategy)
    eng.set_option("bam", 1)
    eng.set_option("deflate", 1)
    try:
        reads, maf, st, text = run.simulate(c.seqset, rng_mode=capi.RNG_REPLAY, replay_draws=draws, replay_starts=starts)
    finally:
        eng.set_option("bam", 0)
        eng.set_option("deflate", 0)
    raw = b"".join(pl for _, pl in B.bgzf_blocks(reads))
    got = B.records_to_sam(raw)
    want = c.reads()
    # BAM has no lower-case bases: compare with the reference text upper-cased in the SEQ column only
    def norm(sam):
        rows = []
        for ln in sam.decode().splitlines():
            f = ln.split("\t")
            f[9] = f[9].upper()
            rows.append("\t".join(f))
        return rows
    assert norm(got) == norm(want)


def _genome_with_n_runs(n=160000, seed=3):
    """random ACGT with an N run of 1..400 bases every 9-23 kb: the tiles next to a run take the generic path, the
    rest of the record the staged one"""
    rng = np.random.default_rng(seed)
    g = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)].copy()
    pos = 4000
    while pos < n - 1000:
        g[pos:pos + int(rng.integers(1, 401))] = ord("N")
        pos += int(rng.integers(9000, 23000))
    return g.tobytes()


@pytest.mark.parametrize("method,model", [("qshmm", "QSHMM-RSII.model"), ("errhmm", "ERRHMM-SEQUEL.model")])
@pytest.mark.parametrize("segments", [0, 1])
def test_bam_of_long_reads_across_n_runs_equals_the_sam_text(eng, method, model, segments):
    """PHILOX mode, reads of several tiles each, so that tiles start and end at odd read positions and staged and
    generic tiles share a record: the BAM records decode to the SAM text of the same run, the MAF stream is the same"""
    from tests.golden_util import model_path
    hm = capi.HostModel(capi.load(), capi.host_params(method, pass_num=2, len_mean=6000.0, len_sd=2500.0),
                        model_path(model))
    eng.set_model(hm)
    genome = _genome_with_n_runs()
    eng.set_sequence(genome, 1, [0.0] + [1.0] * 10 + [0.0])
    runs = []
    eng.set_option("segments", segments)
    try:
        for bam in (0, 1):
            eng.set_option("bam", bam)
            reads, maf, _, _ = eng.simulate(2 * len(genome), rng_mode=capi.RNG_PHILOX, seed=21)
            runs.append((reads, maf))
    finally:
        eng.set_option("bam", 0)
        eng.set_option("segments", 1)
    (sam, maf_sam), (bam, maf_bam) = runs
    seqs = [ln.split(b"\t")[9] for ln in sam.splitlines()]
    assert any(b"N" in s and len(s) > 3 * 1024 for s in seqs), "no long record crosses an N run"
    assert B.records_to_sam(bam) == sam
    assert maf_bam == maf_sam
