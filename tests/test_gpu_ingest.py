"""Genome ingest on the device (pbsim_b200/csrc/k0_genome.cuh) against the host reference (tests/ingest_ref.py), base by
base: the upper-cased text, the 2-bit codes, the per-base homopolymer lengths, the exceptional-block bits and the
homopolymer histogram.  Then reads simulated across long N gaps against the oracle, and the driver on a genome with
one.  Run with -m gpu."""
import gzip
import subprocess

import numpy as np
import pytest

import __graft_entry__ as G
from oracle import oracle as O
from pbsim_b200 import capi, simulator
from tests import ingest_ref as R
from tests.golden_util import model_path
from tests.test_ingest_reference_cpu import SHORT_LENGTHS, acgt, mixed_text

pytestmark = pytest.mark.gpu

# bases one pass of k_hp's grid covers (148 * 8 CTAs of 256 threads, 8 bases a thread); longer texts take several
STRIDE = 148 * 8 * 256 * 8
XM_WORD = 32 * 1024  # bases behind one 32-bit word of xm


@pytest.fixture(scope="module")
def eng():
    e = simulator.Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def qs_model():
    return capi.HostModel(capi.load(), capi.host_params("qshmm"), model_path("QSHMM-RSII.model"))


def first_diff(got, want):
    d = np.flatnonzero(got != want)
    return "first difference at %d of %d (got %r, want %r)" % (d[0], len(want), got[d[0]], want[d[0]]) if len(d) else ""


def assert_device_equals(eng, ref):
    n = eng.glen
    ascii = np.empty(n, dtype=np.uint8)
    eng.get_sequence_ascii(ascii.ctypes.data, n)
    pk, hp4, xm = eng.sequence_tables()
    assert np.array_equal(ascii, ref["ascii"]), "ascii: " + first_diff(ascii, ref["ascii"])
    assert np.array_equal(pk, ref["pk"]), "pk word: " + first_diff(pk, ref["pk"])
    hp = R.unpack_hp4(hp4, n)
    assert np.array_equal(hp, ref["hp"]), "hp: " + first_diff(hp, ref["hp"])
    assert np.array_equal(hp4, ref["hp4"]), "hp4 byte (nibble past the end): " + first_diff(hp4, ref["hp4"])
    assert np.array_equal(xm, ref["xm"]), "xm word: " + first_diff(xm, ref["xm"])
    assert eng.hpfreq() == ref["hpfreq"].tolist()
    return xm


# hp 7 is exceptional and hp 11 is not: xm differs from the uniform bias's both ways
HP7_BIAS = [0.0] + [1.0] * 6 + [1.5] + [1.0] * 4


def ingest_each_bias(eng, model, text):
    """uniform bias; the bias a --hp-del-bias 4 prepass gives, ingested the way WgsRun.simulate_sequence does it
    (set_sequence with the prepass bias); and HP7_BIAS.  xm has to follow each set of cells equal to 1"""
    eng.set_sequence(text, 1, R.UNIFORM_BIAS)
    xm_uniform = assert_device_equals(eng, R.ingest(text))
    run = simulator.WgsRun(eng, model, 1.0, hp_del_bias=4.0)
    run.prepass([("s", text)])
    assert [b == 1.0 for b in run.base_bias[1:11]] != [True] * 10
    eng.set_sequence(text, 1, run.base_bias)
    xm_prepass = assert_device_equals(eng, R.ingest(text, run.base_bias))
    eng.set_sequence(text, 1, HP7_BIAS)
    assert_device_equals(eng, R.ingest(text, HP7_BIAS))
    return xm_uniform, xm_prepass


@pytest.mark.parametrize("n", SHORT_LENGTHS + [XM_WORD - 1, XM_WORD, XM_WORD + 1])
def test_short_sequences(eng, qs_model, n):
    rng = np.random.default_rng(100 + n)
    for _ in range(4):
        ingest_each_bias(eng, qs_model, mixed_text(rng, n))


def chromosome(n=(48 << 20) - 12345, seed=5):
    """a chromosome-like text: N telomeres and a 3 Mbp N gap, 100 kb N gaps across a k_hp stride boundary, an xm word
    boundary and a 1 Mbp boundary, homopolymers of every length 1..64 and of 1000, 20000 and 65536 bases starting and
    ending on chosen offsets mod 1024, scattered IUPAC codes, and soft-masked stretches over about half the text"""
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    a = letters[rng.integers(0, 4, n)]
    a[rng.integers(0, n, 3000)] = np.frombuffer(b"RYKMSWBDHV", dtype=np.uint8)[rng.integers(0, 10, 3000)]
    residues = [0, 1, 7, 8, 9, 15, 16, 17, 1023]
    pos = 20000
    for L in list(range(1, 65)) + [1000, 20000, 65536]:
        for r in residues:
            for end_aligned in (False, True):
                s = pos + (r - (pos + (L if end_aligned else 0))) % 1024
                k = int(rng.integers(0, 4))
                a[s:s + L] = letters[k]
                a[s - 1] = a[s + L] = letters[(k + 1) % 4]  # the run is exactly L long
                pos = s + L + 2 + int(rng.integers(0, 20000))
    assert pos < n - 20000
    gaps = [(0, 10000), (n - 10000, 10000), (20000003, 3000000),
            (3 * STRIDE - 50001, 100000),      # across a stride boundary
            (5 * STRIDE, 100003),              # from one
            (7 * STRIDE - 100000, 100000),     # up to one
            (300 * XM_WORD - 7, 100000),       # across an xm word boundary
            (12 * 2 ** 20 - 65537, 100001),    # across a 1 Mbp (1024-block) boundary
            (30 * 2 ** 20 + 1, 65537)]
    for s, L in gaps:
        a[s:s + L] = ord("N")
    lens = rng.integers(1, 6000, n // 3000 + 16)
    masked = np.repeat(np.arange(len(lens)) & 1, lens)[:n].astype(bool)
    a[masked] |= 0x20  # lower case (every byte here is an upper-case letter)
    return a.tobytes()


def test_chromosome_like_sequence(eng, qs_model):
    text = chromosome()
    xm_uniform, xm_prepass = ingest_each_bias(eng, qs_model, text)
    ones = lambda xm: int(np.unpackbits(xm.view(np.uint8)).sum())  # noqa: E731
    assert ones(xm_prepass) > 2 * ones(xm_uniform)


def test_synthetic_sequence(eng):
    n = 2 * STRIDE + 12345  # not a multiple of 16; three passes of k_hp's grid
    eng.set_synthetic_sequence(n, 1, 77)
    ascii = np.empty(n, dtype=np.uint8)
    eng.get_sequence_ascii(ascii.ctypes.data, n)
    assert set(np.unique(ascii).tolist()) == set(b"ACGT")
    assert_device_equals(eng, R.ingest(ascii.tobytes()))


def make_set(rng, strategy):
    """empty and one-base sequences, lower-case first bases, an all-N transcript, runs that touch the boundaries
    between sequences, and a long sequence holding a 100 kb N gap"""
    trans = strategy == "trans"
    long_seq = bytearray(acgt(rng, 300000))
    long_seq[123457:223457] = b"N" * 100000
    fixed = [(b"", 0, 0), (b"a", 0, 0), (b"G", 0, 0), (b"t", 0, 0), (b"N" * 50, 2, 1),
             (b"aaaaaaaaaaaaAAAAAAAAAAAAAAAAAAAAA", 1, 1), (b"AAAAAAAAAAAAAAAAAAAAAAAAAAAAA", 1, 0),
             (b"ccccccccccccccccccccccccccccccccCCCC", 0, 3), (b"CCCCCCCCCCCCCCCCCCCCCC", 2, 2),
             (bytes(long_seq), 1, 2), (b"", 0, 0)]
    rnd = [(mixed_text(rng, int(L)), int(p), int(m)) for L, p, m in
           zip(rng.integers(21, 3000, 40), rng.integers(0, 4, 40), rng.integers(0, 4, 40))]
    out = []
    for k, (s, p, m) in enumerate(fixed + rnd):
        if trans and p + m and len(s) <= 20:
            continue
        if not trans and not s:
            continue
        out.append(("t%d" % k, p, m, s))
    return out


@pytest.mark.parametrize("strategy", ["trans", "templ"])
@pytest.mark.parametrize("method,model", [("qshmm", "QSHMM-RSII.model"), ("errhmm", "ERRHMM-ONT-HQ.model")])
def test_sequence_sets(eng, strategy, method, model):
    rng = np.random.default_rng(len(strategy) + len(method))
    seqset = make_set(rng, strategy)
    seqs = [x[3] for x in seqset]
    weights = [x[1] + x[2] for x in seqset] if strategy == "trans" else None
    keep_first = not (strategy == "trans" and method == "qshmm")
    eng.set_model(capi.HostModel(capi.load(), capi.host_params(method), model_path(model)))
    eng.set_seqset(strategy, seqset, R.UNIFORM_BIAS)
    ref = R.ingest_set(seqs, keep_first, weights)
    assert_device_equals(eng, ref)
    starts = np.cumsum([0] + [len(s) for s in seqs])[:-1]
    firsts = [int(at) for at, s in zip(starts, seqs) if s[:1].islower()]
    assert len(firsts) >= 3
    assert all(chr(ref["ascii"][at]).islower() == keep_first for at in firsts)
    bias = capi.hp_del_bias(eng.L, 4.0, eng.hpfreq())
    eng.set_seqset(strategy, seqset, bias)
    assert_device_equals(eng, R.ingest_set(seqs, keep_first, weights, bias))


def test_what_is_refused(eng):
    """N runs of any length are accepted (every N base has hp 1); a run of another letter is refused once it is
    twice the walk cap long.  Between 65537 and about 65543 bases the outcome depends on alignment: nothing is pinned"""
    rng = np.random.default_rng(3)
    for L in (65537, 200000, 5000000):
        for lead in (1000, 1003, 1007):
            text = acgt(rng, lead) + b"N" * L + acgt(rng, 1001)
            eng.set_sequence(text, 1, R.UNIFORM_BIAS)
            ref = R.ingest(text)
            assert np.all(ref["hp"][lead:lead + L] == 1)
            assert_device_equals(eng, ref)
    for lead in (1000, 1001, 1007, 1008):
        text = acgt(rng, lead - 1) + b"G" + b"A" * 65536 + b"G" + acgt(rng, 1000)
        eng.set_sequence(text, 1, R.UNIFORM_BIAS)
        assert_device_equals(eng, R.ingest(text))
    with pytest.raises(simulator.EngineError, match="homopolymer longer than 65536 bases"):
        eng.set_sequence(acgt(rng, 999) + b"G" + b"T" * 131072 + b"G" + acgt(rng, 1000), 1, R.UNIFORM_BIAS)


def gapped_genome():
    """1.5 Mbp: a 70 kb N gap at the start, a 150 kb one inside, and 20 kb homopolymers elsewhere"""
    rng = np.random.default_rng(21)
    g = bytearray(acgt(rng, 1500000))
    g[:70000] = b"N" * 70000
    g[700000:850000] = b"N" * 150000
    g[300000:320000] = b"A" * 20000
    g[1100000:1120000] = b"c" * 20000
    return bytes(g), [(0, 70000), (700000, 850000)]


@pytest.mark.parametrize("segments", [1, 0])
@pytest.mark.parametrize("method,model,okw", [("qshmm", "QSHMM-ONT.model", dict(len_mean=10000.0)),
                                              ("errhmm", "ERRHMM-ONT-HQ.model", {})])
def test_simulation_across_long_gaps_equals_oracle(eng, method, model, okw, segments):
    genome, gaps = gapped_genome()
    depth, seed = 3.0, 17
    o = O.Oracle(method, model_path(model), **okw)
    o.rng_philox(seed)
    o.set_sequence(genome, 1)
    oreads, omaf, ost = o.simulate_wgs(depth)
    hm = capi.HostModel(capi.load(), capi.host_params(method, **okw), model_path(model))
    run = simulator.WgsRun(eng, hm, depth)
    eng.set_option("segments", segments)
    try:
        reads, maf, st, text = run.simulate_sequence(genome, 1, rng_mode=capi.RNG_PHILOX, seed=seed)
    finally:
        eng.set_option("segments", 1)
    assert reads == oreads
    assert maf == omaf
    assert text == O.format_stats(ost, 1)
    windows = []
    for blk in maf.split(b"\n\n")[:-1]:
        f = blk.split(b"\n")[1].split()
        windows.append((int(f[2]), int(f[2]) + int(f[3])))
    for lo, hi in gaps:
        assert any(lo <= a and b <= hi for a, b in windows), "no read inside the gap [%d, %d)" % (lo, hi)
        assert any(a < lo < b or a < hi < b for a, b in windows), "no read across an edge of [%d, %d)" % (lo, hi)


def test_driver_on_a_genome_with_a_long_n_gap(tmp_path):
    """pbsim --genome on a two-record FASTA, one record holding a 100 kb N gap (PHILOX draws): exit 0, reads equal
    the oracle's"""
    from oracle import refrun as RR
    rng = np.random.default_rng(8)
    first = bytearray(acgt(rng, 250000))
    first[80000:180000] = b"N" * 100000
    contigs = [("chrA", bytes(first)), ("chrB", acgt(rng, 60000))]
    RR.write_fasta(str(tmp_path / "genome.fa"), contigs)
    depth, seed, mp = 2, 5, model_path("QSHMM-RSII.model")
    exe = G.build_driver()
    p = subprocess.run([exe, "--strategy", "wgs", "--method", "qshmm", "--qshmm", mp, "--genome", "genome.fa",
                        "--depth", str(depth), "--seed", str(seed), "--prefix", "out"],
                       cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()
    o = O.Oracle("qshmm", mp)
    o.rng_philox(seed)
    for i, (_, s) in enumerate(contigs, start=1):
        o.set_sequence(s, i)
        reads, _, _ = o.simulate_wgs(depth)
        assert gzip.open(tmp_path / ("out_%04d.fq.gz" % i), "rb").read() == reads, "reads of record %d" % i
