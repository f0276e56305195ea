"""CPU checks of the host ingest reference (tests/ingest_ref.py) against the oracle's independent restatement of
get_genome_seq (Oracle.set_sequence, then hp() and seq_upper()), before tests/test_gpu_ingest.py compares the device
ingest with it."""
import numpy as np
import pytest

from oracle import oracle as O
from pbsim_b200 import capi
from tests import hostsim_util as H
from tests import ingest_ref as R
from tests.golden_util import model_path

SHORT_LENGTHS = [1, 2, 7, 8, 9, 15, 16, 17, 1023, 1024, 1025]


def mixed_text(rng, n, alphabet=b"ACGTACGTacgtNnRYKMSWBDHVry"):
    """runs of random letters (A, C, G, T, N, IUPAC codes, either case) with lengths 1..20: runs of the same letter in
    both cases, adjacent runs of the same letter and runs across sequence ends all occur"""
    letters = np.frombuffer(alphabet, dtype=np.uint8)
    k = n // 2 + 2
    run_len = np.minimum(rng.geometric(0.3, k), 20)
    return np.repeat(letters[rng.integers(0, len(letters), k)], run_len)[:n].tobytes()


def acgt(rng, n):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)].tobytes()


@pytest.fixture(scope="module")
def oracle():
    o = O.Oracle("qshmm", model_path("QSHMM-RSII.model"))
    yield o
    o.close()


def check_against_oracle(o, text):
    o.set_sequence(text, 1)
    r = R.ingest(text)
    assert r["ascii"].tobytes() == o.seq_upper()
    want = o.hp()
    assert np.array_equal(r["hp"], want)
    assert np.array_equal(r["hpfreq"], np.bincount(want, minlength=12))
    return r


@pytest.mark.parametrize("n", SHORT_LENGTHS)
def test_short_sequences_equal_oracle(oracle, n):
    rng = np.random.default_rng(n)
    for _ in range(20):
        check_against_oracle(oracle, mixed_text(rng, n))


@pytest.mark.parametrize("gap", [70000, 1000000])
def test_long_n_gaps_equal_oracle(oracle, gap):
    rng = np.random.default_rng(gap)
    for text in (b"N" * gap, acgt(rng, 5000) + b"N" * gap + acgt(rng, 3001),
                 b"n" * 7 + b"N" * gap + b"nA", acgt(rng, 1) + b"N" * (gap - 1)):
        r = check_against_oracle(oracle, text)
        assert np.all(r["hp"][r["ascii"] == ord("N")] == 1)


@pytest.mark.parametrize("L", [10, 11, 12, 13, 14, 65536])
def test_homopolymers_equal_oracle(oracle, L):
    rng = np.random.default_rng(L)
    run = bytearray(b"A" * L)
    run[L // 2:] = b"a" * (L - L // 2)  # a run of one letter in both cases is one run after upper-casing
    r = check_against_oracle(oracle, acgt(rng, 999) + b"C" + bytes(run) + b"G" + acgt(rng, 1000))
    h = r["hp"][1000:1000 + L]
    assert np.all(h == (L if L <= 11 else 10 if (L - 11) % 2 else 11))


def test_lower_case_and_iupac_equal_oracle(oracle):
    rng = np.random.default_rng(7)
    check_against_oracle(oracle, mixed_text(rng, 300000, alphabet=b"acgtnrykmswbdhvACGTNRYKMSWBDHV"))


@pytest.mark.parametrize("opt", [2.0, 4.0, 7.25])
def test_wgs_hpfreq_through_the_prepass_equals_oracle(opt):
    """the --hp-del-bias prepass over several sequences: the bias the product's host front end derives from the
    reference's hpfreq equals the oracle's; cell 0 carries the summed hpfreq[11] bit for bit"""
    rng = np.random.default_rng(int(opt * 100))
    contigs = [mixed_text(rng, int(n)) for n in rng.integers(1, 40000, 5)] + [b"N" * 70000 + b"TTTTTTTTTTTTT"]
    o = O.Oracle("qshmm", model_path("QSHMM-RSII.model"), hp_del_bias=opt)
    o.hp_bias_prepass(contigs)
    hpfreq = sum(R.ingest(s)["hpfreq"] for s in contigs)
    assert hpfreq[0] == 0 and hpfreq[11] > 0
    bias = capi.hp_del_bias(H.lib(), opt, hpfreq)
    assert bias[1:11] == o.bias()[1:11].tolist()
    assert np.array([bias[0]]).view(np.int64)[0] == hpfreq[11]


@pytest.mark.parametrize("keep_first", [False, True])
def test_set_ingest_equals_oracle_per_sequence(oracle, keep_first):
    """a set is its sequences one after the other: runs end at sequence boundaries.  With keep_first a lower-case
    first base stays lower case and is a run of its own; the oracle sees it as a byte that equals no other"""
    rng = np.random.default_rng(11 + keep_first)
    seqs = [b"", b"a", b"A", b"aAAAA", b"AAAA", b"NNNN", b"nNNN", b"c", b"CCCCCCCCCCCCC", b""] + \
        [mixed_text(rng, int(n)) for n in rng.integers(1, 3000, 30)]
    weights = rng.integers(0, 5, len(seqs))
    r = R.ingest_set(seqs, keep_first, weights)
    at, want_freq = 0, np.zeros(12, dtype=np.int64)
    for s, w in zip(seqs, weights):
        if s:
            first_kept = keep_first and s[:1].islower()
            oracle.set_sequence((b"\x01" + s[1:]) if first_kept else s, 1)
            up = oracle.seq_upper()
            if first_kept:
                up = s[:1] + up[1:]
            want = oracle.hp()
            assert r["ascii"][at:at + len(s)].tobytes() == up
            assert np.array_equal(r["hp"][at:at + len(s)], want)
            want_freq += w * np.bincount(want, minlength=12)
            assert r["pk"][at // 16] >> (2 * (at % 16)) & 3 == (R._CODE[up[0]] if not first_kept else 0)
        at += len(s)
    assert np.array_equal(r["hpfreq"], want_freq)


def test_layouts_by_hand():
    """pk, hp4 and xm bit positions on hand-made text"""
    text = bytearray(b"ACGT" * 10000)
    text[3] = ord("G")                              # "ACGG": hp 2 at bases 2 and 3
    text[5 * 1024 + 100:5 * 1024 + 111] = b"G" * 11  # hp 11, and bias[11] = 0 in the uniform bias: block 5
    text[7 * 1024:7 * 1024 + 8] = b"acgtacgt"       # lower case is upper-cased: block 7 stays clear
    text[9 * 1024:9 * 1024 + 12] = b"C" * 12        # hp 10, bias 1: block 9 stays clear
    text[33 * 1024 + 5] = ord("R")                  # block 33: word 1, bit 1
    text[39999] = ord("N")                          # the last block, 64 bases long: word 1, bit 7
    r = R.ingest(bytes(text))
    assert len(r["pk"]) == 2500 and len(r["hp4"]) == 20000 and len(r["xm"]) == 2
    assert r["pk"][0] == 0xE4E4E4A4 and r["pk"][1] == 0xE4E4E4E4
    assert r["pk"][2499] == 0x24E4E4E4  # the N packs as 0
    assert r["hp4"][0] == 0x11 and r["hp4"][1] == 0x22 and r["hp4"][2] == 0x11
    assert r["xm"][0] == 1 << 5 and r["xm"][1] == (1 << 1) | (1 << 7)
    assert np.array_equal(R.unpack_hp4(r["hp4"], len(text)), r["hp"])
