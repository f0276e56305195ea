"""TEST CODE: an independent MAF -> SAM converter for option "align" / `--align sam`, and a checker of its records.

Plain Python over the text the reference writes (a reads stream and a MAF stream); it shares no code with the engine.
The record is the one include/pbsim_cuda.h documents for option "align"."""

_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def parse_maf(maf):
    """MAF text -> [(src, start, size, src_size, ref_row, read_name, strand, read_row)] in file order"""
    out = []
    for block in maf.split(b"\n\n"):
        if not block:
            continue
        lines = block.split(b"\n")
        assert lines[0] == b"a", block[:40]
        f = lines[1].split()
        g = lines[2].split()
        assert f[0] == b"s" and g[0] == b"s" and f[4] == b"+"
        out.append((f[1], int(f[2]), int(f[3]), int(f[5]), f[6], g[1], g[4], g[6]))
    return out


def parse_reads(reads, pass_num):
    """FASTQ (pass_num 1) or headerless SAM text -> [(name, seq, qual)]"""
    out = []
    if pass_num == 1:
        lines = reads.split(b"\n")
        for i in range(0, len(lines) - 1, 4):
            out.append((lines[i][1:], lines[i + 1], lines[i + 3]))
    else:
        for line in reads.split(b"\n"):
            if line:
                f = line.split(b"\t")
                out.append((f[0], f[9], f[10]))
    return out


def column_ops(ref_row, read_row):
    """'=' 'X' 'I' 'D' per MAF column"""
    ops = bytearray()
    for a, b in zip(ref_row, read_row):
        ops.append(73 if a == 45 else (68 if b == 45 else (61 if a == b else 88)))  # I D = X
    return bytes(ops)


def runs(ops):
    out = []
    for o in ops:
        if out and out[-1][0] == o:
            out[-1][1] += 1
        else:
            out.append([o, 1])
    return out


def to_sam(reads, maf, pass_num, rname=None, sample=False):
    """The alignment lines of one stream pair.  rname: RNAME of every record (WGS); None: the MAF row's source name
    (transcript / template sets).  sample: --method sample, whose MAF start field is the window's first base even when a
    minus-strand read stopped before its window was used up: the true leftmost base is rlen - size further right."""
    blocks = parse_maf(maf)
    recs = parse_reads(reads, pass_num)
    assert len(blocks) == len(recs)
    lines = []
    for (src, start, size, _, ref_row, _, strand, read_row), (name, seq, qual) in zip(blocks, recs):
        minus = strand == b"-"
        ops = column_ops(ref_row, read_row)
        mx = [i for i, o in enumerate(ops) if o in b"=X"]
        sam_seq = read_row.replace(b"-", b"")
        assert sam_seq == (seq[::-1].translate(_COMP) if minus else seq)
        sam_qual = qual[::-1] if minus else qual
        if not sam_seq:
            sam_seq = sam_qual = b"*"
        if not mx:
            lines.append(b"\t".join([name, b"4", b"*", b"0", b"0", b"*", b"*", b"0", b"0", sam_seq, sam_qual,
                                     b"NM:i:0"]))
            continue
        lo, hi = mx[0], mx[-1] + 1
        pos = start + (max(0, len(seq) - size) if sample and minus else 0) + ops[:lo].count(b"D") + 1
        cigar = b""
        if ops[:lo].count(b"I"):
            cigar += b"%dS" % ops[:lo].count(b"I")
        cigar += b"".join(b"%d%c" % (n, o) for o, n in runs(ops[lo:hi]))
        if ops[hi:].count(b"I"):
            cigar += b"%dS" % ops[hi:].count(b"I")
        nm = sum(1 for o in ops[lo:hi] if o != 61)
        lines.append(b"\t".join([name, b"16" if minus else b"0", rname if rname is not None else src, b"%d" % pos,
                                 b"60", cigar, b"*", b"0", b"0", sam_seq, sam_qual, b"NM:i:%d" % nm]))
    return b"".join(x + b"\n" for x in lines)


def parse_cigar(cigar):
    out, n = [], 0
    for ch in cigar:
        if 48 <= ch <= 57:
            n = n * 10 + ch - 48
        else:
            out.append((chr(ch), n))
            n = 0
    return out


def check_record(line, ref_row, read_row, genome):
    """One alignment line against the MAF block it came from; genome: the text POS counts in (compared without case:
    sets keep a lower-case first base)."""
    f = line.split(b"\t")
    assert len(f) == 12 and f[11].startswith(b"NM:i:")
    ops = column_ops(ref_row, read_row)
    if f[1] == b"4":
        assert f[5] == b"*" and f[3] == b"0" and not any(o in b"=X" for o in ops)
        return
    cig = parse_cigar(f[5])
    seq = f[9] if f[9] != b"*" else b""
    assert sum(n for op, n in cig if op in "=XIS") == len(seq), "CIGAR query length != len(SEQ)"
    assert all(n > 0 for _, n in cig)
    assert all(a != b for (a, _), (b, _) in zip(cig, cig[1:])), "adjacent runs of one op"
    assert cig[0][0] in "=XS" and cig[-1][0] in "=XS" and all(op != "S" for op, _ in cig[1:-1])
    # the walk rebuilds the MAF rows between the first and last = / X column
    mx = [i for i, o in enumerate(ops) if o in b"=X"]
    lo, hi = mx[0], mx[-1] + 1
    g = int(f[3]) - 1
    q = cig[0][1] if cig[0][0] == "S" else 0
    rr, qr, cols, nm = bytearray(), bytearray(), bytearray(), 0
    for op, n in cig:
        if op == "S":
            continue
        cols += op.encode() * n
        if op in "=XD":
            rr += genome[g:g + n]
            g += n
        else:
            rr += b"-" * n
        if op in "=XI":
            qr += seq[q:q + n]
            q += n
        else:
            qr += b"-" * n
        if op != "=":
            nm += n
    assert bytes(rr).upper() == ref_row[lo:hi].upper() and bytes(qr) == read_row[lo:hi], \
        "CIGAR walk does not rebuild the MAF rows"
    for op, a, b in zip(bytes(cols), ref_row[lo:hi], read_row[lo:hi]):
        if op in b"=X":
            assert (a == b) == (op == 61), "%c column with bytes %c %c" % (op, a, b)
    assert int(f[11][5:]) == nm
    # outside: the clipped insertions and the dropped deletions, which sit right in front of POS
    lead, trail = ops[:lo], ops[hi:]
    assert (cig[0][1] if cig[0][0] == "S" else 0) == lead.count(b"I")
    assert (cig[-1][1] if cig[-1][0] == "S" else 0) == trail.count(b"I")
    nd = lead.count(b"D")
    assert ref_row[:lo].replace(b"-", b"").upper() == genome[int(f[3]) - 1 - nd:int(f[3]) - 1].upper()
