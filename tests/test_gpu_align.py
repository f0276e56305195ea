"""-m gpu: option "align" (SAM alignment lines in the second stream).  The engine's lines must equal the independent
converter of tests/aln_util.py applied to the reference's own files (replay mode) and to the engine's and the oracle's
MAF runs (PHILOX mode), byte for byte; the reads stream must not change."""
import zlib

import numpy as np
import pytest

from oracle import oracle as O
from pbsim_b200 import capi, simulator
from tests import aln_util as A
from tests.golden_util import Case, SampleCase, SetCase, case_names, sample_case_names, set_case_names
from tests.gpu_util import engine_model

pytestmark = pytest.mark.gpu


def _name(hdr):
    return hdr.split()[0].encode()


@pytest.fixture(scope="module")
def eng():
    e = simulator.Engine(0)
    e.set_option("align", 1)
    yield e
    e.close()


def _wgs(c, eng, mode, oracle_out=None, **kw):
    """run_case_on_gpu with every sequence named by its FASTA header's first word"""
    run = simulator.WgsRun(eng, engine_model(c), c.depth, hp_del_bias=c.okw.get("hp_del_bias", 1.0))
    if c.okw.get("hp_del_bias", 1.0) != 1.0:
        run.prepass(c.contigs)
    res = []
    if mode == "replay":
        draws = O.glibc_rand(c.seed, c.ndraws)
        starts = np.concatenate([[0], c.marks[:-1]]).astype(np.int64)
        pos = 0
        for i, (hdr, s) in enumerate(c.contigs, start=1):
            n = len(oracle_out[i - 1]["info"])
            end = int(starts[pos + n]) if pos + n < len(starts) else c.ndraws
            res.append(run.simulate_sequence(s, i, name=_name(hdr), rng_mode=capi.RNG_REPLAY, replay_draws=draws[:end],
                                             replay_starts=starts[pos:pos + n], **kw))
            pos += n
    else:
        for i, (hdr, s) in enumerate(c.contigs, start=1):
            res.append(run.simulate_sequence(s, i, name=_name(hdr), rng_mode=capi.RNG_PHILOX, seed=c.seed, **kw))
    return res


@pytest.mark.parametrize("name", case_names())
def test_replay_equals_converted_reference(eng, name):
    c = Case(name)
    out, _ = c.run_oracle("glibc")
    for i, (reads, sam, _, text) in enumerate(_wgs(c, eng, "replay", out), start=1):
        assert reads == c.reads(i), "reads stream changed, seq %d" % i
        assert sam == A.to_sam(c.reads(i), c.maf(i), c.pass_num, rname=_name(c.contigs[i - 1][0])), "seq %d" % i
        assert text == c.stats_blocks[i]


@pytest.mark.parametrize("name", set_case_names())
def test_replay_sets_equal_converted_reference(eng, name):
    c = SetCase(name)
    draws = O.glibc_rand(c.seed, c.ndraws)
    starts = np.concatenate([[0], c.marks[:-1]]).astype(np.int64)
    run = simulator.SetRun(eng, capi.HostModel(capi.load(), capi.host_params(c.method, **c.okw), c.model), c.strategy,
                           hp_del_bias=c.okw.get("hp_del_bias", 1.0))
    reads, sam, _, _ = run.simulate(c.seqset, rng_mode=capi.RNG_REPLAY, replay_draws=draws, replay_starts=starts)
    assert reads == c.reads()
    assert sam == A.to_sam(c.reads(), c.maf(), c.pass_num)


@pytest.mark.parametrize("name", sample_case_names())
def test_replay_sample_equals_converted_reference(name):
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
            reads, sam, _, _ = run.simulate_sequence(s, i, name=_name(hdr), rng_mode=capi.RNG_REPLAY,
                                                     replay_draws=draws[:end], replay_starts=starts[pos:pos + n])
            pos += n
            assert reads == c.reads(i)
            assert sam == A.to_sam(c.reads(i), c.maf(i), 1, rname=_name(hdr), sample=True), "seq %d" % i
    finally:
        eng.close()


@pytest.mark.parametrize("name", case_names())
def test_philox_equals_converted_oracle(eng, name):
    c = Case(name)
    out, _ = c.run_oracle("philox")
    for i, ((reads, sam, _, _), o) in enumerate(zip(_wgs(c, eng, "philox"), out), start=1):
        assert reads == o["reads"]
        assert sam == A.to_sam(o["reads"], o["maf"], c.pass_num, rname=_name(c.contigs[i - 1][0])), "seq %d" % i


@pytest.mark.parametrize("name", ["qs_rsii_quirks", "err_sequel_multipass", "qs_delheavy_uniform"])
@pytest.mark.parametrize("segments", [0, 1])
@pytest.mark.parametrize("batch", [1, 7, 64])
@pytest.mark.parametrize("pipeline", [0, 1, 2])
def test_philox_equals_converted_maf_run(name, segments, batch, pipeline):
    """the engine's own --align maf run converted, over segments, batch sizes and pipeline modes"""
    c = Case(name)
    e = simulator.Engine(0)
    try:
        e.set_option("segments", segments)
        e.set_option("pipeline", pipeline)
        maf_run = _wgs(c, e, "philox", batch_reads=batch)
        e.set_option("align", 1)
        sam_run = _wgs(c, e, "philox", batch_reads=batch)
    finally:
        e.close()
    for i, (m, s) in enumerate(zip(maf_run, sam_run), start=1):
        assert s[0] == m[0]
        assert s[1] == A.to_sam(m[0], m[1], c.pass_num, rname=_name(c.contigs[i - 1][0]))


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
    eng.set_sequence_name(_name(hdr))
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
    assert b"".join(ms) == A.to_sam(out[0]["reads"], out[0]["maf"], 1, rname=_name(hdr))


def _members(blob):
    out = []
    while blob:
        d = zlib.decompressobj(16 + zlib.MAX_WBITS)
        out.append(d.decompress(blob))
        assert d.eof
        blob = d.unused_data
    return b"".join(out)


@pytest.mark.parametrize("name", ["qs_rsii_basic", "err_sequel_multipass"])
def test_deflate_members_inflate_to_the_lines(eng, name):
    c = Case(name)
    plain = _wgs(c, eng, "philox")
    eng.set_option("deflate", 1)
    try:
        packed = _wgs(c, eng, "philox")
    finally:
        eng.set_option("deflate", 0)
    for p, z in zip(plain, packed):
        assert _members(z[0]) == p[0]
        assert _members(z[1]) == p[1]


def test_fuzz_seeds_equal_converted_oracle(eng):
    """24 further seeds, spread over the golden setups"""
    for seed in range(24):
        c = Case(case_names()[seed % len(case_names())])
        c.seed = 1000 + seed
        out, _ = c.run_oracle("philox")
        for i, ((reads, sam, _, _), o) in enumerate(zip(_wgs(c, eng, "philox"), out), start=1):
            assert sam == A.to_sam(o["reads"], o["maf"], c.pass_num, rname=_name(c.contigs[i - 1][0])), (seed, i)


def test_misuse_fails_loudly_and_leaves_the_engine_usable():
    c = Case("qs_rsii_basic")
    e = simulator.Engine(0)
    try:
        e.set_model(engine_model(c))
        hdr, s = c.contigs[0]
        e.set_sequence(s, 1, [0.0] + [1.0] * 10 + [0.0])
        e.set_option("align", 1)
        with pytest.raises(simulator.EngineError, match="set_sequence_name"):
            e.begin(1000, rng_mode=capi.RNG_PHILOX, seed=1)
        with pytest.raises(simulator.EngineError, match="whitespace"):
            e.set_sequence_name("chr 1")
        e.set_sequence_name(_name(hdr))
        e.set_option("bam", 1)
        with pytest.raises(simulator.EngineError, match="align and bam"):
            e.begin(1000, rng_mode=capi.RNG_PHILOX, seed=1)
        e.set_option("bam", 0)
        e.set_sequence(s, 1, [0.0] + [1.0] * 10 + [0.0])  # forgets the name
        with pytest.raises(simulator.EngineError, match="set_sequence_name"):
            e.begin(1000, rng_mode=capi.RNG_PHILOX, seed=1)
        e.set_sequence_name(_name(hdr))
        reads, sam, _, _ = e.simulate(int(c.depth * len(s)), rng_mode=capi.RNG_PHILOX, seed=c.seed)
        assert sam == A.to_sam(reads, _maf_of(c, s), 1, rname=_name(hdr))
    finally:
        e.close()


def _maf_of(c, s):
    e = simulator.Engine(0)
    try:
        e.set_model(engine_model(c))
        e.set_sequence(s, 1, [0.0] + [1.0] * 10 + [0.0])
        return e.simulate(int(c.depth * len(s)), rng_mode=capi.RNG_PHILOX, seed=c.seed)[1]
    finally:
        e.close()


def _cli(c, wd, extra, genome_text=None):
    import gzip
    import subprocess

    import __graft_entry__ as G
    exe = G.build_driver()
    with gzip.open(c.dir + "/genome.fa.gz", "rb") as f:
        (wd / "genome.fa").write_bytes(genome_text if genome_text is not None else f.read())
    args = [exe, "--strategy", "wgs", "--method", c.method, "--" + c.method, c.model, "--genome", "genome.fa",
            "--depth", str(c.depth), "--seed", str(c.seed)] + list(c.meta["extra_args"]) + ["--prefix", "out"] + extra
    p = subprocess.run(args, cwd=wd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()


@pytest.mark.parametrize("name,extra", [("qs_rsii_basic", []), ("err_onthq_basic", []),
                                        ("qs_rsii_multipass", ["--gzip", "host"])])
def test_cli_align_sam_equals_converted_maf_run(name, extra, tmp_path):
    """--align sam on a FASTA whose headers carry descriptions: header + converter(the --align maf run's files); the
    reads files do not change"""
    import gzip
    c = Case(name)
    fa = b"".join(b">%s described here\n%s\n" % (b"chr%d" % i, s) for i, (_, s) in enumerate(c.contigs, start=1))
    (tmp_path / "maf").mkdir()
    (tmp_path / "sam").mkdir()
    _cli(c, tmp_path / "maf", extra, fa)
    _cli(c, tmp_path / "sam", extra + ["--align", "sam"], fa)
    ext = ".fq.gz" if c.pass_num == 1 else ".sam.gz"
    for i, (_, s) in enumerate(c.contigs, start=1):
        reads = gzip.open(tmp_path / "maf" / ("out_%04d%s" % (i, ext)), "rb").read()
        assert gzip.open(tmp_path / "sam" / ("out_%04d%s" % (i, ext)), "rb").read() == reads
        assert not (tmp_path / "sam" / ("out_%04d.maf.gz" % i)).exists()
        maf = gzip.open(tmp_path / "maf" / ("out_%04d.maf.gz" % i), "rb").read()
        if c.pass_num > 1:
            reads = reads[reads.index(b"PM:SEQUELII\n") + len(b"PM:SEQUELII\n"):]
        head = b"@HD\tVN:1.6\tSO:unknown\n@SQ\tSN:chr%d\tLN:%d\n@PG\tID:pbsim\tPN:pbsim\n" % (i, len(s))
        got = gzip.open(tmp_path / "sam" / ("out_%04d.aln.sam.gz" % i), "rb").read()
        assert got == head + A.to_sam(reads, maf, c.pass_num, rname=b"chr%d" % i)
