"""TEST CODE: an independent reader and writer of aligned BAM for option "align_bam" / `--align-encoding bam`.

Plain Python from the SAM spec (sections 4.1, 4.2, 4.2.2, 5.3); it shares no code with the engine.  The reader prints
every record as the SAM line option "align" writes (tests/aln_util.py) and checks the fields a SAM line does not show:
block_size, l_read_name, bin, the fixed mate fields, the pad nibble and the tag types.  The writer turns such a SAM line
into its record, for the tests that run without a GPU."""
import struct

from tests import bam_util as B

NT16 = B.NT16
OPS = "MIDNSHP=X"
MAX_OPS = 65535


def reg2bin(beg, end):
    end -= 1
    for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return first + (beg >> shift)
    return 0


def int_type(v):
    """the smallest unsigned type, as htslib's SAM parser picks it for a non-negative value"""
    return "C" if v <= 255 else ("S" if v <= 65535 else "I")


def _ref_span(ops):
    return sum(n for op, n in ops if op in "MDN=X")


def parse_cigar(text):
    out, n = [], 0
    for ch in text:
        if ch.isdigit():
            n = n * 10 + int(ch)
        else:
            out.append((ch, n))
            n = 0
    return out


def encode_record(line, names):
    """one SAM line of option "align" (no newline) -> its BAM record; names: the @SQ names in order"""
    f = line.split(b"\t")
    assert len(f) == 12 and f[11].startswith(b"NM:i:")
    qname, flag, rname, pos, mapq, cigar, seq, qual = f[0], int(f[1]), f[2], int(f[3]), int(f[4]), f[5], f[9], f[10]
    ref_id = -1 if rname == b"*" else names.index(rname)
    ops = [] if cigar == b"*" else parse_cigar(cigar.decode())
    seq = b"" if seq == b"*" else seq
    qual = b"" if qual == b"*" else qual
    span = _ref_span(ops)
    bin_ = 4680 if flag & 4 else reg2bin(pos - 1, pos - 1 + span)
    words = [n << 4 | OPS.index(op) for op, n in ops]
    cg = len(words) > MAX_OPS
    field = [len(seq) << 4 | 4, span << 4 | 3] if cg else words
    body = struct.pack("<iiBBHHHIiii", ref_id, pos - 1, len(qname) + 1, mapq, bin_, len(field), flag, len(seq), -1, -1, 0)
    body += qname + b"\0" + struct.pack("<%dI" % len(field), *field)
    packed = bytearray((len(seq) + 1) // 2)
    for i, ch in enumerate(seq):
        packed[i >> 1] |= NT16.index(chr(ch).upper()) << (0 if i & 1 else 4)
    body += bytes(packed) + bytes(q - 33 for q in qual)
    nm = int(f[11][5:])
    t = int_type(nm)
    body += b"NM" + t.encode() + struct.pack({"C": "<B", "S": "<H", "I": "<I"}[t], nm)
    if cg:
        body += b"CGBI" + struct.pack("<I%dI" % len(words), len(words), *words)
    return struct.pack("<I", len(body)) + body


def upper_seq(sam):
    """SAM lines with SEQ upper-cased: what they decode to from BAM, which has no lower-case bases (sets keep a
    lower-case first base)"""
    out = []
    for ln in sam.split(b"\n"):
        if ln:
            f = ln.split(b"\t")
            f[9] = f[9].upper()
            out.append(b"\t".join(f) + b"\n")
    return b"".join(out)


def encode_records(sam, names):
    return b"".join(encode_record(ln, names) for ln in sam.split(b"\n") if ln)


def decode_records(raw, names, stats=None):
    """BAM alignment records (no file header) -> the SAM lines of option "align"; stats (a dict) counts the records
    that were unmapped, empty or held their CIGAR in a CG tag"""
    lines, p = [], 0
    while p < len(raw):
        (block_size,) = struct.unpack_from("<I", raw, p)
        rec = raw[p + 4:p + 4 + block_size]
        assert len(rec) == block_size, "record runs past the end"
        p += 4 + block_size
        ref_id, pos, l_name, mapq, bin_, n_cigar, flag, l_seq, nref, npos, tlen = struct.unpack_from("<iiBBHHHIiii", rec)
        assert (nref, npos, tlen) == (-1, -1, 0)
        q = 32
        name = rec[q:q + l_name - 1]
        assert rec[q + l_name - 1] == 0 and b"\0" not in name
        q += l_name
        words = list(struct.unpack_from("<%dI" % n_cigar, rec, q))
        q += 4 * n_cigar
        packed = rec[q:q + (l_seq + 1) // 2]
        q += (l_seq + 1) // 2
        seq = "".join(NT16[(packed[i >> 1] >> (0 if i & 1 else 4)) & 15] for i in range(l_seq))
        if l_seq & 1:
            assert packed[-1] & 15 == 0, "pad nibble is not 0"
        qual = bytes(x + 33 for x in rec[q:q + l_seq]).decode()
        q += l_seq
        assert rec[q:q + 2] == b"NM", "NM must be the first tag"
        t = chr(rec[q + 2])
        nm, q = B._int_tag(t, rec, q + 3)
        assert t == int_type(nm), "NM:%s holds %d" % (t, nm)
        ops = [(OPS[w & 15], w >> 4) for w in words]
        if q < len(rec):
            assert rec[q:q + 4] == b"CGBI", "unexpected tag %r" % rec[q:q + 4]
            (cnt,) = struct.unpack_from("<I", rec, q + 4)
            real = [(OPS[w & 15], w >> 4) for w in struct.unpack_from("<%dI" % cnt, rec, q + 8)]
            q += 8 + 4 * cnt
            assert cnt > MAX_OPS and ops == [("S", l_seq), ("N", _ref_span(real))], "CG placeholder %r" % ops
            ops = real
            if stats is not None:
                stats["cg"] = stats.get("cg", 0) + 1
        assert q == len(rec), "bytes after the tags"
        mapped = not flag & 4
        if mapped:
            assert ref_id >= 0 and pos >= 0 and mapq == 60
            assert bin_ == reg2bin(pos, pos + _ref_span(ops)), "bin"
        else:
            assert (ref_id, pos, mapq, bin_, ops) == (-1, -1, 0, 4680, [])
        if stats is not None:
            stats["unmapped"] = stats.get("unmapped", 0) + (not mapped)
            stats["empty"] = stats.get("empty", 0) + (l_seq == 0)
            stats["records"] = stats.get("records", 0) + 1
        cigar = "".join("%d%s" % (n, op) for op, n in ops) if ops else "*"
        lines.append("\t".join([name.decode(), str(flag), names[ref_id] if ref_id >= 0 else "*", str(pos + 1), str(mapq),
                                cigar, "*", "0", "0", seq or "*", qual or "*", "NM:i:%d" % nm]) + "\n")
    return "".join(lines).encode()


def parse_header(raw):
    """BAM file header -> (header text, [(name, length)], size of the header in bytes)"""
    assert raw[:4] == b"BAM\x01"
    (l_text,) = struct.unpack_from("<I", raw, 4)
    text = raw[8:8 + l_text]
    (n_ref,) = struct.unpack_from("<I", raw, 8 + l_text)
    p, refs = 12 + l_text, []
    for _ in range(n_ref):
        (l_name,) = struct.unpack_from("<I", raw, p)
        name = raw[p + 4:p + 4 + l_name - 1]
        assert raw[p + 4 + l_name - 1] == 0
        (l_ref,) = struct.unpack_from("<I", raw, p + 4 + l_name)
        refs.append((name.decode(), l_ref))
        p += 8 + l_name
    sq = [(ln.split("\t")[1][3:], int(ln.split("\t")[2][3:])) for ln in text.decode().splitlines() if ln.startswith("@SQ")]
    assert sq == refs, "n_ref / names / lengths disagree with the @SQ lines"
    return text, refs, p


def parse_aln_bam(blob, stats=None):
    """a whole .aln.bam -> (header text, [(name, length)], SAM lines, number of BGZF blocks of the header); checks the
    blocks (BSIZE, CRC, ISIZE) and the end-of-file block"""
    blocks = B.bgzf_blocks(blob)
    assert blocks[-1] == (28, b""), "missing BGZF end-of-file block"
    raw = b"".join(pl for _, pl in blocks)
    text, refs, n = parse_header(raw)
    hdr_blocks, acc = 0, 0
    while acc < n:
        acc += len(blocks[hdr_blocks][1])
        hdr_blocks += 1
    return text, refs, decode_records(raw[n:], [r for r, _ in refs], stats), hdr_blocks
