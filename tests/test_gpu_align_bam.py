"""-m gpu: option "align_bam" (BAM alignment records in the second stream) and `--align-encoding bam`.  The records
are decoded by the independent reader of tests/aln_bam_util.py and must give exactly the SAM lines of option "align"
(SEQ upper-cased: BAM has no lower-case bases): the converter's lines of the reference's own files in replay mode, the
engine's own lines in PHILOX mode.  The reads stream must not change."""
import gzip
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from pbsim_b200 import capi, simulator
from tests import aln_bam_util as AB
from tests import aln_util as A
from tests import bam_util as B
from tests.golden_util import Case, SampleCase, SetCase, case_names, model_path, sample_case_names, set_case_names
from tests.gpu_util import engine_model
from tests.test_gpu_align import _cli, _name, _wgs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = simulator.Engine(0)
    e.set_option("align", 1)
    e.set_option("align_bam", 1)
    yield e
    e.close()


def _set_names(c):
    return [n if isinstance(n, str) else n.decode() for n, _, _, _ in c.seqset]


@pytest.mark.parametrize("name", case_names())
def test_replay_decodes_to_converted_reference(eng, name):
    c = Case(name)
    out, _ = c.run_oracle("glibc")
    for i, (reads, bam, _, text) in enumerate(_wgs(c, eng, "replay", out), start=1):
        rname = _name(c.contigs[i - 1][0])
        assert reads == c.reads(i), "reads stream changed, seq %d" % i
        want = A.to_sam(c.reads(i), c.maf(i), c.pass_num, rname=rname)
        assert AB.decode_records(bam, [rname.decode()]) == AB.upper_seq(want), "seq %d" % i
        assert text == c.stats_blocks[i]


@pytest.mark.parametrize("name", set_case_names())
def test_replay_sets_decode_to_converted_reference(eng, name):
    c = SetCase(name)
    draws = O.glibc_rand(c.seed, c.ndraws)
    starts = np.concatenate([[0], c.marks[:-1]]).astype(np.int64)
    run = simulator.SetRun(eng, capi.HostModel(capi.load(), capi.host_params(c.method, **c.okw), c.model), c.strategy,
                           hp_del_bias=c.okw.get("hp_del_bias", 1.0))
    reads, bam, _, _ = run.simulate(c.seqset, rng_mode=capi.RNG_REPLAY, replay_draws=draws, replay_starts=starts)
    assert reads == c.reads()
    assert AB.decode_records(bam, _set_names(c)) == AB.upper_seq(A.to_sam(c.reads(), c.maf(), c.pass_num))


@pytest.mark.parametrize("name", sample_case_names())
def test_replay_sample_decodes_to_converted_reference(name):
    """--method sample, whose minus-strand reads may leave window bases unused (the POS correction)"""
    c = SampleCase(name)
    o = O.Oracle("sample", None, **c.okw)
    o.rng_glibc(c.seed)
    if c.okw.get("hp_del_bias", 1.0) != 1.0:
        o.hp_bias_prepass([s for _, s in c.contigs])
    counts = []
    for i, (_, s) in enumerate(c.contigs, start=1):
        o.set_sequence(s, i)
        o.simulate_sample(c.depth, c.pool)
        counts.append(len(o.readinfo()))
    eng = simulator.Engine(0)
    try:
        eng.set_option("align", 1)
        eng.set_option("align_bam", 1)
        run = simulator.WgsRun(eng, capi.HostModel(capi.load(), capi.host_params("sample", **c.okw), None), c.depth,
                               c.okw.get("hp_del_bias", 1.0))
        eng.set_pool(c.pool)
        if c.okw.get("hp_del_bias", 1.0) != 1.0:
            run.prepass(c.contigs)
        draws = O.glibc_rand(c.seed, c.ndraws)
        starts = np.concatenate([[0], c.marks[:-1]]).astype(np.int64)
        pos = 0
        for i, (hdr, s) in enumerate(c.contigs, start=1):
            n = counts[i - 1]
            end = int(starts[pos + n]) if pos + n < len(starts) else c.ndraws
            reads, bam, _, _ = run.simulate_sequence(s, i, rng_mode=capi.RNG_REPLAY, replay_draws=draws[:end],
                                                     replay_starts=starts[pos:pos + n])
            pos += n
            assert reads == c.reads(i)
            want = A.to_sam(c.reads(i), c.maf(i), 1, rname=_name(hdr), sample=True)
            assert AB.decode_records(bam, [_name(hdr).decode()]) == AB.upper_seq(want), "seq %d" % i
    finally:
        eng.close()


@pytest.mark.parametrize("name", ["qs_rsii_quirks", "err_sequel_multipass"])
@pytest.mark.parametrize("segments", [0, 1])
@pytest.mark.parametrize("batch", [1, 7, 64])
@pytest.mark.parametrize("pipeline", [0, 1, 2])
def test_philox_decodes_to_the_sam_lines_of_the_same_run(name, segments, batch, pipeline):
    c = Case(name)
    e = simulator.Engine(0)
    try:
        e.set_option("segments", segments)
        e.set_option("pipeline", pipeline)
        e.set_option("align", 1)
        sam_run = _wgs(c, e, "philox", batch_reads=batch)
        e.set_option("align_bam", 1)
        bam_run = _wgs(c, e, "philox", batch_reads=batch)
    finally:
        e.close()
    for i, (s, b) in enumerate(zip(sam_run, bam_run), start=1):
        assert b[0] == s[0]
        assert AB.decode_records(b[1], [_name(c.contigs[i - 1][0]).decode()]) == s[1], "seq %d" % i


@pytest.mark.parametrize("name", ["err_sequel_multipass", "qs_rsii_multipass"])
def test_bam_reads_with_bam_alignments(name):
    """bam + align + align_bam: the reads are those of a bam-only run, the alignments decode to the SAM lines of a
    bam = 0 run"""
    c = Case(name)
    e = simulator.Engine(0)
    try:
        e.set_option("align", 1)
        sam_run = _wgs(c, e, "philox")
        e.set_option("align", 0)
        e.set_option("bam", 1)
        bam_only = _wgs(c, e, "philox")
        e.set_option("align", 1)
        e.set_option("align_bam", 1)
        both = _wgs(c, e, "philox")
    finally:
        e.close()
    for i, (s, r, b) in enumerate(zip(sam_run, bam_only, both), start=1):
        assert b[0] == r[0], "BAM reads stream changed, seq %d" % i
        assert AB.decode_records(b[1], [_name(c.contigs[i - 1][0]).decode()]) == s[1], "seq %d" % i


@pytest.mark.parametrize("name,bam", [("qs_rsii_basic", 0), ("err_sequel_multipass", 1)])
def test_deflate_writes_bgzf_blocks_of_the_records(eng, name, bam):
    c = Case(name)
    eng.set_option("bam", bam)
    try:
        plain = _wgs(c, eng, "philox")
        eng.set_option("deflate", 1)
        packed = _wgs(c, eng, "philox")
    finally:
        eng.set_option("deflate", 0)
        eng.set_option("bam", 0)
    for p, z in zip(plain, packed):
        blocks = B.bgzf_blocks(z[1])  # BSIZE, CRC and ISIZE of every block
        assert len(blocks) > 0 and b"".join(pl for _, pl in blocks) == p[1]
        if bam:
            assert b"".join(pl for _, pl in B.bgzf_blocks(z[0])) == p[0]


def test_device_delivery(eng):
    from tests.test_gpu_parity import _device_bytes
    c = Case("qs_rsii_basic")
    out, _ = c.run_oracle("philox")
    run = simulator.WgsRun(eng, engine_model(c), c.depth)
    hdr, s = c.contigs[0]
    bias = list(run.base_bias)
    eng.set_sequence(s, 1, bias)
    bias[0] = float(np.array([eng.hpfreq()[11]], dtype=np.int64).view(np.float64)[0])
    eng.update_bias(bias)
    eng.begin(int(c.depth * len(s)), rng_mode=capi.RNG_PHILOX, seed=c.seed, batch_reads=13)
    rs, ms = [], []
    while True:
        ch = eng.next_chunk(device=True)
        if ch is None:
            break
        rs.append(_device_bytes(ch.reads, ch.reads_bytes))
        ms.append(_device_bytes(ch.maf, ch.maf_bytes))
    eng.end()
    del run
    assert b"".join(rs) == out[0]["reads"]
    want = A.to_sam(out[0]["reads"], out[0]["maf"], 1, rname=_name(hdr))
    assert AB.decode_records(b"".join(ms), [_name(hdr).decode()]) == AB.upper_seq(want)


def _both_encodings(hm, genome, quota, seed):
    e = simulator.Engine(0)
    try:
        e.set_model(hm)
        e.set_sequence(genome, 1, [0.0] + [1.0] * 10 + [0.0])
        e.set_sequence_name("chr1")
        e.set_option("align", 1)
        reads_s, sam, _, _ = e.simulate(quota, rng_mode=capi.RNG_PHILOX, seed=seed)
        e.set_option("align_bam", 1)
        reads_b, bam, _, _ = e.simulate(quota, rng_mode=capi.RNG_PHILOX, seed=seed)
    finally:
        e.close()
    assert reads_b == reads_s
    return sam, bam


def _random_genome(n, seed):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[np.random.default_rng(seed).integers(0, 4, n)].tobytes()


def test_more_than_65535_ops_use_the_cg_tag():
    """reads of ~400 kb at accuracy 0.75 have far more than 65,535 runs"""
    hm = capi.HostModel(capi.load(), capi.host_params("qshmm", accuracy_mean=0.75, accuracy_mean_set=True,
                                                      len_min=300000, len_max=1000000, len_mean=400000.0, len_sd=0.0),
                        model_path("QSHMM-RSII.model"))
    genome = _random_genome(2000000, 5)
    sam, bam = _both_encodings(hm, genome, 1200000, 11)
    st = {}
    assert AB.decode_records(bam, ["chr1"], st) == sam
    assert st.get("cg", 0) >= 1, st


@pytest.mark.parametrize("ratio", [(0, 50, 50), (0, 100, 0)])
def test_unmapped_records(ratio):
    """--method sample with a pool of 1- and 2-base quality strings of '!' (error probability 1) and insertions and
    deletions only: many reads have no = / X column and are written unmapped (refID -1, pos -1, MAPQ 0, bin 4680, no
    CIGAR, FLAG 4), of both length parities.  Their records decode to the engine's own SAM lines, which
    equal the converter's lines of the oracle's run.  An empty read (rlen 0) cannot arise, since every read is at least
    len_min >= 1 bases long: tests/test_align_bam_cpu.py is the only coverage of that record."""
    genome = _random_genome(20000, 6)
    pool = [b"!" * (1 + i % 2) for i in range(400)]
    okw = dict(ratio=ratio, len_min=1, len_max=4)
    o = O.Oracle("sample", None, **okw)
    o.rng_philox(3)
    o.set_sequence(genome, 1)
    oreads, omaf, _ = o.simulate_sample(0.2, pool)
    runs = []
    e = simulator.Engine(0)
    try:
        e.set_option("align", 1)
        for align_bam in (0, 1):
            e.set_option("align_bam", align_bam)
            run = simulator.WgsRun(e, capi.HostModel(capi.load(), capi.host_params("sample", **okw), None), 0.2)
            e.set_pool(pool)
            runs.append(run.simulate_sequence(genome, 1, name=b"chr1", rng_mode=capi.RNG_PHILOX, seed=3))
    finally:
        e.close()
    (reads_s, sam, _, _), (reads_b, bam, _, _) = runs
    assert reads_s == reads_b == oreads
    assert sam == A.to_sam(oreads, omaf, 1, rname=b"chr1", sample=True)
    st = {}
    assert AB.decode_records(bam, ["chr1"], st) == sam
    unmapped = [ln.split(b"\t") for ln in sam.splitlines() if ln.split(b"\t")[1] == b"4"]
    assert st["unmapped"] == len(unmapped) > 100
    assert {len(f[9]) % 2 for f in unmapped} == {0, 1}


def test_misuse_fails_loudly_and_leaves_the_engine_usable():
    c = Case("qs_rsii_basic")
    e = simulator.Engine(0)
    try:
        e.set_model(engine_model(c))
        hdr, s = c.contigs[0]
        e.set_sequence(s, 1, [0.0] + [1.0] * 10 + [0.0])
        e.set_option("align_bam", 1)
        with pytest.raises(simulator.EngineError, match="align_bam needs option align"):
            e.begin(1000, rng_mode=capi.RNG_PHILOX, seed=1)
        e.set_option("align", 1)
        e.begin(int(c.depth * len(s)), rng_mode=capi.RNG_PHILOX, seed=c.seed)
        with pytest.raises(simulator.EngineError, match="align_bam cannot change during a run"):
            e.set_option("align_bam", 0)
        e.end()
        reads, bam, _, _ = e.simulate(int(c.depth * len(s)), rng_mode=capi.RNG_PHILOX, seed=c.seed)
        e.set_option("align_bam", 0)
        e.set_sequence_name(_name(hdr))
        reads_s, sam, _, _ = e.simulate(int(c.depth * len(s)), rng_mode=capi.RNG_PHILOX, seed=c.seed)
    finally:
        e.close()
    assert reads == reads_s and AB.decode_records(bam, [_name(hdr).decode()]) == sam


def _files(d, stem):
    return sorted(p.name for p in d.iterdir() if p.name.startswith(stem))


@pytest.mark.parametrize("name,host", [("qs_rsii_basic", False), ("err_onthq_basic", False),
                                       ("qs_rsii_multipass", True)])
def test_cli_aln_bam_decodes_to_the_aln_sam_file(name, host, tmp_path):
    """.aln.bam = header and body of the --align sam run's .aln.sam.gz (multi-pass: that run needs --gzip host); the
    reads files are those of a run without --align (multi-pass: the .bam of a --gzip gpu run)"""
    c = Case(name)
    fa = b"".join(b">%s described here\n%s\n" % (b"chr%d" % i, s) for i, (_, s) in enumerate(c.contigs, start=1))
    for d in ("plain", "sam", "bam"):
        (tmp_path / d).mkdir()
    _cli(c, tmp_path / "plain", [], fa)
    _cli(c, tmp_path / "sam", ["--align", "sam"] + (["--gzip", "host"] if host else []), fa)
    _cli(c, tmp_path / "bam", ["--align", "sam", "--align-encoding", "bam"], fa)
    ext = ".fq.gz" if c.pass_num == 1 else ".bam"
    for i in range(1, len(c.contigs) + 1):
        stem = "out_%04d" % i
        assert (tmp_path / "bam" / (stem + ext)).read_bytes() == (tmp_path / "plain" / (stem + ext)).read_bytes()
        assert not (tmp_path / "bam" / (stem + ".aln.sam.gz")).exists()
        assert not (tmp_path / "bam" / (stem + ".maf.gz")).exists()
        text, refs, body, _ = AB.parse_aln_bam((tmp_path / "bam" / (stem + ".aln.bam")).read_bytes())
        want = gzip.open(tmp_path / "sam" / (stem + ".aln.sam.gz"), "rb").read()
        assert want.startswith(text) and body == AB.upper_seq(want[len(text):])
        assert refs == [("chr%d" % i, len(c.contigs[i - 1][1]))]


def _set_cli(tmp_path, d, strategy, method, model, inp, extra):
    import __graft_entry__ as G
    exe = G.build_driver()
    args = [exe, "--strategy", strategy, "--method", method, "--" + method, model,
            "--transcript" if strategy == "trans" else "--template", str(inp), "--seed", "7", "--prefix", "out"] + extra
    p = subprocess.run(args, cwd=tmp_path / d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()


def _big_transcript_table(path, n=3000):
    """n transcripts with 60-character ids, a few of them expressed: the @SQ lines alone are ~240 kB"""
    rng = np.random.default_rng(9)
    with open(path, "w") as f:
        for t in range(n):
            seq = _random_genome(int(rng.integers(200, 3000)), t).decode()
            plus, minus = (3, 2) if t % 97 == 0 else (0, 0)
            f.write("tr%058d\t%d\t%d\t%s\n" % (t, plus, minus, seq))


@pytest.mark.parametrize("which", ["tr_qs_rsii_basic", "tm_qs_rsii_basic", "big_trans"])
def test_cli_sets_aln_bam_decodes_to_the_aln_sam_file(which, tmp_path):
    if which == "big_trans":
        inp = tmp_path / "input.txt"
        _big_transcript_table(inp)
        strategy, method, model, extra = "trans", "qshmm", model_path("QSHMM-RSII.model"), []
    else:
        c = SetCase(which)
        inp = tmp_path / "input.txt"
        with gzip.open(c.dir + "/input.txt.gz", "rb") as f:
            inp.write_bytes(f.read())
        strategy, method, model, extra = c.strategy, c.method, c.model, list(c.meta["extra_args"])
    for d in ("plain", "sam", "bam"):
        (tmp_path / d).mkdir()
    _set_cli(tmp_path, "plain", strategy, method, model, inp, extra)
    _set_cli(tmp_path, "sam", strategy, method, model, inp, extra + ["--align", "sam"])
    _set_cli(tmp_path, "bam", strategy, method, model, inp, extra + ["--align", "sam", "--align-encoding", "bam"])
    ext = ".fq.gz" if (tmp_path / "plain" / "out.fq.gz").exists() else ".bam"
    assert (tmp_path / "bam" / ("out" + ext)).read_bytes() == (tmp_path / "plain" / ("out" + ext)).read_bytes()
    text, refs, body, hdr_blocks = AB.parse_aln_bam((tmp_path / "bam" / "out.aln.bam").read_bytes())
    want = gzip.open(tmp_path / "sam" / "out.aln.sam.gz", "rb").read()
    assert want.startswith(text) and body == AB.upper_seq(want[len(text):])
    if which == "big_trans":
        assert len(refs) == 3000 and hdr_blocks > 1
