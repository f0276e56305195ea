"""Host reference of genome ingest: what get_genome_seq (pbsim.cpp:1032-1065) and the per-sequence ingest of the
transcript / template sets leave behind, in the layout the engine keeps in HBM (pbsim_b200/csrc/k0_genome.cuh):
upper-cased text, 2-bit codes (pk), per-base homopolymer lengths (hp), one exceptional bit per 1024-base block (xm) and
the homopolymer histogram (hpfreq).  Plain numpy on run boundaries; the tests check it against the oracle first."""
import numpy as np

XM_BLOCK = 1024
UNIFORM_BIAS = [0.0] + [1.0] * 10 + [0.0]

_CODE = np.zeros(256, dtype=np.uint8)
_ACGT = np.zeros(256, dtype=bool)
for _k, _c in enumerate(b"ACGT"):
    _CODE[_c] = _k
    _ACGT[_c] = True


def as_u8(text):
    return np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else np.asarray(text, np.uint8)


def upper(text):
    """toupper in the C locale"""
    a = as_u8(text).copy()
    low = (a >= ord("a")) & (a <= ord("z"))
    a[low] -= 32
    return a


def hp_of_runs(a, seq_starts=None):
    """per-base homopolymer length of upper-cased text: a run of L equal bytes gives L for L <= 11, else 10 if L - 11
    is odd and 11 if it is even (the reference's counter: nnum > 11 -> 10); every base of an N run gets 1.
    seq_starts: first base of every sequence of a set; runs end there."""
    n = len(a)
    if n == 0:
        return np.zeros(0, dtype=np.uint8)
    brk = np.zeros(n, dtype=bool)
    brk[0] = True
    brk[1:] = a[1:] != a[:-1]
    if seq_starts is not None:
        s = np.asarray(seq_starts, dtype=np.int64)
        brk[s[s < n]] = True
    starts = np.flatnonzero(brk)
    L = np.diff(np.append(starts, n))
    h = np.where(L <= 11, L, np.where((L - 11) & 1, 10, 11)).astype(np.uint8)
    h[a[starts] == ord("N")] = 1
    return np.repeat(h, L)


def pack_codes(a):
    """pk: A=0 C=1 G=2 T=3, anything else 0; base i at bits 2*(i%16) of word i/16; bits past the end 0"""
    n = len(a)
    c = np.zeros(-(-n // 16) * 16, dtype=np.uint32)
    c[:n] = _CODE[a]
    return (c.reshape(-1, 16) << (2 * np.arange(16, dtype=np.uint32))).sum(axis=1, dtype=np.uint32)


def pack_hp4(hp):
    """hp4: base i in the low nibble of byte i/2 when i is even, the high nibble when odd"""
    h = np.zeros(-(-len(hp) // 2) * 2, dtype=np.uint8)
    h[:len(hp)] = hp
    return h[0::2] | (h[1::2] << 4)


def unpack_hp4(hp4, n):
    return np.stack([hp4 & 15, hp4 >> 4], axis=1).reshape(-1)[:n]


def exceptional_bits(a, hp, bias):
    """xm: block b is set iff one of its bases is not A, C, G or T, or has an hp h with bias[h] != 1 (bias[0] counts
    as 1: hp 0 never occurs); block b at bit b%32 of word b/32, bits past the last block 0"""
    n = len(a)
    one = np.array([b == 1.0 for b in bias], dtype=bool)
    one[0] = True
    bad = np.zeros(-(-n // XM_BLOCK) * XM_BLOCK, dtype=bool)
    bad[:n] = ~_ACGT[a] | ~one[hp]
    blocks = bad.reshape(-1, XM_BLOCK).any(axis=1)
    bits = np.zeros(-(-len(blocks) // 32) * 32, dtype=bool)
    bits[:len(blocks)] = blocks
    return np.packbits(bits, bitorder="little").view("<u4").astype(np.uint32)


def _tables(a, hp, weight, bias):
    # float64 weights: the sums of the test sets stay far below 2^53, where they are exact
    hpfreq = np.bincount(hp, weights=weight, minlength=12).astype(np.int64)
    return dict(ascii=a, hp=hp, pk=pack_codes(a), hp4=pack_hp4(hp), xm=exceptional_bits(a, hp, bias), hpfreq=hpfreq)


def ingest(text, bias=UNIFORM_BIAS):
    """one genome sequence (get_genome_seq)"""
    a = upper(text)
    return _tables(a, hp_of_runs(a), None, bias)


def ingest_set(seqs, keep_first, weights=None, bias=UNIFORM_BIAS):
    """a transcript or template set, concatenated.  keep_first: every sequence's first base keeps its case (all but
    simulate_by_qshmm_trans upper-case from the second base, pbsim.cpp:3330, :4474, :5049 against :2774).
    weights: per sequence, how often its bases count in hpfreq (transcripts: plus + minus reads, :2714-2718)."""
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    raw = as_u8(b"".join(seqs))
    a = upper(raw)
    if keep_first:
        f = starts[lens > 0]
        a[f] = raw[f]
    hp = hp_of_runs(a, starts)
    w = None if weights is None else np.repeat(np.asarray(weights, dtype=np.float64), lens)
    return _tables(a, hp, w, bias)
