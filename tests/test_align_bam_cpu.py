"""Aligned BAM without a GPU: the reader and writer of tests/aln_bam_util.py against each other on the SAM lines of all
golden runs and on hand-built records, and the driver's refusals of --align-encoding."""
import struct
import subprocess

import pytest

from tests import aln_bam_util as AB
from tests import aln_util as A
from tests.golden_util import Case, SampleCase, SetCase, case_names, sample_case_names, set_case_names


def _golden_sam():
    for name in case_names():
        c = Case(name)
        for i, (hdr, _) in enumerate(c.contigs, start=1):
            rname = hdr.split()[0].encode()
            yield name, [rname], A.to_sam(c.reads(i), c.maf(i), c.pass_num, rname=rname)
    for name in set_case_names():
        c = SetCase(name)
        yield name, [s[0].encode() if isinstance(s[0], str) else s[0] for s in c.seqset], A.to_sam(c.reads(), c.maf(),
                                                                                                  c.pass_num)
    for name in sample_case_names():
        c = SampleCase(name)
        for i, (hdr, _) in enumerate(c.contigs, start=1):
            rname = hdr.split()[0].encode()
            yield name, [rname], A.to_sam(c.reads(i), c.maf(i), 1, rname=rname, sample=True)


def test_round_trip_of_every_golden_run():
    runs = set()
    minus = lines = 0
    for name, names, sam in _golden_sam():
        runs.add(name)
        raw = AB.encode_records(sam, names)
        assert AB.decode_records(raw, [n.decode() for n in names]) == AB.upper_seq(sam), name
        lines += sam.count(b"\n")
        minus += sum(1 for ln in sam.split(b"\n") if ln and ln.split(b"\t")[1] == b"16")
    assert len(runs) == 23 and lines > 2000 and minus > 500


def _line(name, flag, rname, pos, cigar, seq, qual, nm):
    return b"\t".join([name, b"%d" % flag, rname, b"%d" % pos, b"0" if flag & 4 else b"60", cigar, b"*", b"0", b"0", seq,
                       qual, b"NM:i:%d" % nm])


def _decode_one(rec, names=("chr1",)):
    st = {}
    got = AB.decode_records(rec, list(names), st)
    return got, st


def test_unmapped_record():
    line = _line(b"S1_7", 4, b"*", 0, b"*", b"ACG", b"!#%", 0)
    rec = AB.encode_record(line, [b"chr1"])
    ref_id, pos, l_name, mapq, bin_, n_cigar, flag, l_seq = struct.unpack_from("<iiBBHHHI", rec, 4)
    assert (ref_id, pos, mapq, bin_, n_cigar, flag, l_seq) == (-1, -1, 0, 4680, 0, 4, 3)
    got, st = _decode_one(rec)
    assert got == line + b"\n" and st["unmapped"] == 1


def test_empty_read():
    line = _line(b"S1_8", 4, b"*", 0, b"*", b"*", b"*", 0)
    rec = AB.encode_record(line, [b"chr1"])
    assert struct.unpack_from("<I", rec, 20)[0] == 0  # l_seq
    assert len(rec) == 4 + 32 + len(b"S1_8") + 1 + 4  # no CIGAR, SEQ, QUAL; NM:C
    got, st = _decode_one(rec)
    assert got == line + b"\n" and st["empty"] == 1


def test_odd_length_minus_strand_read():
    line = _line(b"S1_9/3/0", 16, b"chr1", 70001, b"1S2=1X1D1=", b"TACGN", b"+,-./", 2)
    rec = AB.encode_record(line, [b"chr1"])
    _, pos, _, _, bin_, n_cigar, flag, l_seq = struct.unpack_from("<iiBBHHHI", rec, 4)
    assert (pos, n_cigar, flag, l_seq) == (70000, 5, 16, 5)
    assert bin_ == AB.reg2bin(70000, 70005) == 4681 + (70000 >> 14)
    packed = rec[4 + 32 + 9 + 20:4 + 32 + 9 + 20 + 3]
    assert packed == bytes([0x81, 0x24, 0xF0])  # T A, C G, N + pad nibble 0
    got, _ = _decode_one(rec)
    assert got == line + b"\n"
    bad = bytearray(rec)
    bad[4 + 32 + 9 + 20 + 2] |= 1
    with pytest.raises(AssertionError, match="pad nibble"):
        AB.decode_records(bytes(bad), ["chr1"])


def test_more_than_65535_ops_go_to_a_cg_tag():
    n = 70000
    cigar = b"5S" + b"".join((b"2=", b"1X", b"1=", b"1I")[i % 4] for i in range(n - 2)) + b"3S"
    ops = AB.parse_cigar(cigar.decode())
    assert len(ops) == n
    qlen = sum(k for op, k in ops if op in "=XIS")
    span = sum(k for op, k in ops if op in "=XD")
    nm = sum(k for op, k in ops if op in "XID")
    seq = (b"ACGT" * qlen)[:qlen]
    line = _line(b"S1_1", 0, b"chr1", 12345, cigar, seq, b"5" * qlen, nm)
    rec = AB.encode_record(line, [b"chr1"])
    _, pos, l_name, _, bin_, n_cigar = struct.unpack_from("<iiBBHH", rec, 4)
    assert n_cigar == 2 and bin_ == AB.reg2bin(pos, pos + span)
    kS, mN = struct.unpack_from("<II", rec, 4 + 32 + l_name)
    assert (kS, mN) == (qlen << 4 | 4, span << 4 | 3)
    assert rec.index(b"NM") < rec.index(b"CGBI")
    got, st = _decode_one(rec)
    assert got == line + b"\n" and st["cg"] == 1


def _driver(tmp_path, extra):
    import __graft_entry__ as G
    G.build_engine()
    exe = G.build_driver()
    (tmp_path / "g.fa").write_text(">s\n" + "ACGT" * 100 + "\n")
    return subprocess.run([exe, "--strategy", "wgs", "--method", "qshmm", "--qshmm", "x.model", "--genome", "g.fa"] + extra,
                          cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120)


@pytest.mark.parametrize("extra,msg", [
    (["--align", "sam", "--align-encoding", "cram"], "ERROR (align-encoding: cram): Acceptable value: text, bam.\n"),
    (["--align-encoding", "bam"], "ERROR: --align-encoding bam needs --align sam.\n"),
    (["--align", "maf", "--align-encoding", "bam"], "ERROR: --align-encoding bam needs --align sam.\n"),
])
def test_driver_rejects_bad_align_encodings(tmp_path, extra, msg):
    p = _driver(tmp_path, extra)
    assert p.returncode != 0
    assert p.stderr.decode().endswith(msg)


def test_driver_rejects_bam_alignments_with_host_gzip(tmp_path):
    p = _driver(tmp_path, ["--align", "sam", "--align-encoding", "bam", "--gzip", "host"])
    assert p.returncode != 0
    err = p.stderr.decode()
    assert err.startswith("ERROR: --align-encoding bam needs --gzip gpu") and "BGZF" in err
