"""The alignment-line converter of tests/aln_util.py on the reference's own outputs (every golden run: WGS, transcript
and template sets, --method sample, multi-pass): each record's CIGAR walked over the sequence from POS must rebuild
the MAF block it came from.  The GPU tests then hold the engine's option "align" to this converter byte for byte."""
import pytest

from tests import aln_util as A
from tests.golden_util import Case, SampleCase, SetCase, case_names, sample_case_names, set_case_names


def _check_stream(reads, maf, pass_num, genomes, rname_of, sample=False):
    """genomes: src name (bytes) -> sequence text; rname_of: RNAME for to_sam (None: the MAF source name)"""
    sam = A.to_sam(reads, maf, pass_num, rname=rname_of, sample=sample)
    lines = sam.split(b"\n")[:-1]
    blocks = A.parse_maf(maf)
    assert len(lines) == len(blocks)
    stats = dict(minus=0, clipped=0, dropped=0, unmapped=0, moved=0)
    for line, (src, start, size, _, ref_row, _, strand, read_row) in zip(lines, blocks):
        A.check_record(line, ref_row, read_row, genomes[src])
        f = line.split(b"\t")
        stats["minus"] += f[1] == b"16"
        stats["unmapped"] += f[1] == b"4"
        stats["clipped"] += b"S" in f[5]
        if f[1] != b"4":
            ops = A.column_ops(ref_row, read_row)
            lead = ops[:min(i for i, o in enumerate(ops) if o in b"=X")]
            stats["dropped"] += b"D" in lead
            stats["moved"] += int(f[3]) != start + 1 + lead.count(b"D")
    return stats


def _first_word(name):
    return name.split()[0].encode()


@pytest.mark.parametrize("name", case_names())
def test_wgs_goldens(name):
    c = Case(name)
    for i, (hdr, seq) in enumerate(c.contigs, start=1):
        st = _check_stream(c.reads(i), c.maf(i), c.pass_num, {b"ref": seq}, _first_word(hdr))
        assert st["minus"] > 0 and st["moved"] == 0


@pytest.mark.parametrize("name", set_case_names())
def test_set_goldens(name):
    c = SetCase(name)
    genomes = {n.encode(): s for n, _, _, s in c.seqset}
    st = _check_stream(c.reads(), c.maf(), c.pass_num, genomes, None)
    assert st["moved"] == 0


@pytest.mark.parametrize("name", sample_case_names())
def test_sample_goldens(name):
    """--method sample: a minus-strand read that ends on its quality string's length leaves window bases unused, and the
    MAF start field still names the window's first base; the converter moves POS by the unused bases"""
    c = SampleCase(name)
    moved = 0
    for i, (hdr, seq) in enumerate(c.contigs, start=1):
        st = _check_stream(c.reads(i), c.maf(i), 1, {b"ref": seq}, _first_word(hdr), sample=True)
        moved += st["moved"]
    assert moved > 0, "no golden record exercises the start correction"


def test_sample_start_field_is_not_leftmost():
    """without the correction the walk from the MAF start field does not rebuild the reference row"""
    c = SampleCase(sample_case_names()[0])
    _, seq = c.contigs[0]
    sam = A.to_sam(c.reads(1), c.maf(1), 1, rname=b"x", sample=False)
    bad = 0
    for line, blk in zip(sam.split(b"\n"), A.parse_maf(c.maf(1))):
        try:
            A.check_record(line, blk[4], blk[7], seq)
        except AssertionError:
            bad += 1
    assert bad > 0


def test_byte_classes_equal_event_counts():
    """'X' by byte comparison counts exactly the substitutions the reference reports (and I / D its insertions and
    deletions): a substitution never reproduces the reference byte"""
    import re
    for name in case_names():
        c = Case(name)
        if c.pass_num > 1:
            continue
        for i in range(1, len(c.contigs) + 1):
            counts = {b"=": 0, b"X": 0, b"I": 0, b"D": 0}
            for blk in A.parse_maf(c.maf(i)):
                for o in A.column_ops(blk[4], blk[7]):
                    counts[bytes([o])] += 1
            total = sum(len(r[1]) for r in A.parse_reads(c.reads(i), 1))
            block = c.stats_blocks[i]
            for key, op in (("substitution", b"X"), ("insertion", b"I"), ("deletion", b"D")):
                rate = float(re.search(key + r" rate\. : ([0-9.]+)", block).group(1))
                assert abs(counts[op] / total - rate) < 1e-6, (name, i, key)


def test_driver_rejects_a_bad_align_value(tmp_path):
    import subprocess

    import __graft_entry__ as G
    G.build_engine()
    exe = G.build_driver()
    (tmp_path / "g.fa").write_text(">s\n" + "ACGT" * 100 + "\n")
    p = subprocess.run([exe, "--strategy", "wgs", "--method", "qshmm", "--qshmm", "x.model", "--genome", "g.fa",
                        "--align", "bam"], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120)
    assert p.returncode != 0
    assert p.stderr.decode().endswith("ERROR (align: bam): Acceptable value: maf, sam.\n")
