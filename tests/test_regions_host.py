"""The host side of `indelope -r / -R` (bamio.cpp): the region and BED parsers, and idlh_bai_region_run -- the run of BGZF members that holds every record
touching an interval's windows -- checked against the BAM inflated with gzip and walked with struct, independent of the C++ reader."""
import gzip
import struct

import pytest

from indelope_b200 import host
import idl_testutil as util

NAMES = ["chrA", "chrB", "chr:odd", "GL000192.1"]
LENS = [400_000, 50_000, 1_000, 5_000]


def parse(regions=(), bed=None):
    return host.parse_regions(NAMES, LENS, regions, bed)


def test_region_strings():
    assert parse(["chrA:1-10"])[0] == [(0, 10)]                                  # 1-based inclusive -> 0-based half open
    assert parse(["chrA:5"])[0] == [(4, 400_000)]                                # beg to the end of the target
    assert parse(["chrA:5-"])[0] == [(4, 400_000)]
    assert parse(["chrB"])[1] == [(0, 50_000)]                                   # the whole target
    assert parse(["chr:odd"])[2] == [(0, 1_000)]                                 # a name with ':' is a whole target
    assert parse(["chr:odd:2-3"])[2] == [(1, 3)]
    assert parse(["chrA:1,000-2,000"])[0] == [(999, 2000)]                       # thousands commas
    assert parse(["chrA:7-7"])[0] == [(6, 7)]                                    # one base
    assert parse(["chrB:49,990-60,000"])[1] == [(49_989, 50_000)]                # clipped to the target
    # repeated, overlapping, touching and out of order: sorted and merged per target
    r = parse(["chrA:100-200", "chrB:1-5", "chrA:50-99", "chrA:150-300", "chrA:1000-1001"])
    assert r[0] == [(49, 300), (999, 1001)] and r[1] == [(0, 5)]


@pytest.mark.parametrize("bad,msg", [("chrZ:1-10", "no such target"), ("chrZ", "no such target"), ("chrA:0-10", "beg must be >= 1"),
                                     ("chrA:10-5", "end must be >= beg"), ("chrA:x-5", "expected chr"), ("chrA:5-1e3", "expected chr"),
                                     ("chrA:-5", "expected chr"), ("chrA:", "expected chr")])
def test_region_strings_refused(bad, msg):
    with pytest.raises(ValueError, match=msg):
        parse([bad])


def test_bed_files(tmp_path):
    bed = tmp_path / "t.bed"
    bed.write_bytes(b"# comment\r\ntrack name=x\nbrowser position chrA:1-2\n\n"
                    b"chrB\t10\t20\tname\t0\t+\r\n"
                    b"chrA\t300\t400\n"
                    b"chrA 0 10\n"                       # blank-separated columns
                    b"chrA\t350\t500\textra\n"           # overlaps the line before it
                    b"chrA\t500\t600\n"                  # touches it
                    b"chrA\t700\t700\n")                 # empty: selects nothing
    r = parse(bed=str(bed))
    assert r[0] == [(0, 10), (300, 600)] and r[1] == [(10, 20)] and r[2] == []
    # -r and -R together: the union, targets in header order whatever the input order
    r = parse(["chrB:1-3", "chrA:11-12"], bed=str(bed))
    assert r[0] == [(0, 12), (300, 600)] and r[1] == [(0, 3), (10, 20)]


@pytest.mark.parametrize("line,msg", [(b"chrZ\t1\t2", "line 3: target 'chrZ' is not in the BAM header"), (b"chrA\t1", "line 3: expected chrom, start and end"),
                                      (b"chrA\t-1\t5", "line 3: start and end must be"), (b"chrA\t1,0\t50", "line 3: start and end must be"),
                                      (b"chrA\t9\t5", "line 3: end is smaller than start"), (b"chrA\tx\t5", "line 3: start and end must be")])
def test_bed_lines_refused(tmp_path, line, msg):
    bed = tmp_path / "bad.bed"
    bed.write_bytes(b"# header\nchrA\t1\t2\n" + line + b"\n")
    with pytest.raises(ValueError, match=msg):
        parse(bed=str(bed))
    with pytest.raises(ValueError, match="cannot open"):
        parse(bed=str(tmp_path / "missing.bed"))


def test_decoy_targets_are_noted_and_dropped(capfd):
    r = parse(["GL000192.1:1-100", "chrA:1-2"])
    assert r[3] == [] and r[0] == [(0, 2)]
    assert "GL000192.1" in capfd.readouterr().err


# ---- idlh_bai_region_run ----------------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """two targets of ~400 kb (25 linear windows each) and a copy of the file whose second target has no records"""
    d = tmp_path_factory.mktemp("regions")
    ds = util.small_dataset("pr1", chrom_len=400_000, n_events=30, max_indel=40, n_chroms=2, coverage=8)
    fa, bam = str(d / "ref.fa"), str(d / "reads.bam")
    ds.write_fasta(fa)
    ds.write_bam(bam, level=1)
    one = host.Dataset.load_region(fa, bam, "chrS1")
    bam1 = str(d / "one.bam")
    one.write_bam(bam1, level=1)
    return fa, bam, bam1


def _walk(data, at, end):
    """(ref_id, pos, stop, offset) of the records of data[at:end]; stop as bam_endpos counts it"""
    out = []
    while at < end:
        bs, ref_id, pos, l_name, _mapq, _bin, n_cig, flag, _l_seq = struct.unpack_from("<iiiBBHHHi", data, at)
        rlen = 0
        for k in range(n_cig):
            c, = struct.unpack_from("<I", data, at + 36 + l_name + 4 * k)
            if c & 0xf in (0, 2, 3, 7, 8):
                rlen += c >> 4
        if flag & 4 or n_cig == 0 or rlen == 0:
            rlen = 1
        out.append((ref_id, pos, pos + rlen, at)); at += 4 + bs
    assert at == end
    return out


def _all_records(raw):
    whole = gzip.decompress(raw)
    l_text, = struct.unpack_from("<i", whole, 4); at = 8 + l_text
    n_ref, = struct.unpack_from("<i", whole, at); at += 4
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", whole, at); at += 4 + l_name + 4
    return _walk(whole, at, len(whole))


def check_run(bam, raw, allrec, c, beg, end):
    """the run for the windows of [beg, end) as the command line first asks for it, and one window wider on both sides"""
    w0, w1 = ((beg - 1) >> 14) if beg > 0 else 0, ((end - 1) >> 14) + 1
    for a, b in ((w0, w1), (max(w0 - 1, 0), w1 + 1), (w0, w0)):
        sp = host.bai_region_run(bam, c, a, b)
        mine = [r for r in allrec if r[0] == c]
        if sp["empty"]:
            assert not any(r[1] >= (a << 14) - 2000 and r[1] < ((b + 1) << 14) and r[2] > (a << 14) for r in mine)
            continue
        run = raw[sp["file_begin"]:sp["file_end"]]
        inflated = gzip.decompress(run)
        stop_at = len(gzip.decompress(run[:sp["end_member"]])) + sp["end_offset"] if sp["end_member"] else sp["end_offset"]
        recs = _walk(inflated, sp["first_record"], stop_at)                          # starts and ends on record boundaries
        base = len(gzip.decompress(raw[:sp["file_begin"]]))
        got = [(r[0], r[1], r[2], r[3] + base) for r in recs]
        k0 = allrec.index(got[0])
        assert allrec[k0:k0 + len(got)] == got                                     # a contiguous range of the file's records
        inside, before = set(got), [r for r in mine if r[3] < got[0][3]]
        zlo = sp["zone_lo"]
        assert zlo == 0 if (a == 0 or not before) else zlo == (a << 14) + 1
        assert all(r[2] <= zlo - 1 for r in before)                                # nothing in front of the run reaches the zone
        # every record that touches a position of the zone [zlo, start of the run's last record) is in the run ...
        assert {r for r in mine if r[2] >= zlo and r[1] < got[-1][1]} <= inside
        # ... and so is every record that overlaps the interval when the zone covers it
        if zlo <= beg and (sp["to_end"] or got[-1][1] >= end):
            assert {r for r in mine if r[1] < end and r[2] > beg} <= inside
        assert sp["to_end"] == (got[-1] == mine[-1])


@pytest.mark.parametrize("beg,end", [(0, 1), (0, 100), (123_456, 130_000), (16_384, 32_768), (16_383, 16_385), (32_768 * 3, 32_768 * 3 + 1),
                                     (399_000, 400_000), (399_999, 400_000), (0, 400_000), (200_000, 260_000)])
def test_region_run_holds_every_record_of_the_zone(files, beg, end):
    fa, bam, _ = files
    raw = open(bam, "rb").read()
    allrec = _all_records(raw)
    for c in (0, 1):
        check_run(bam, raw, allrec, c, beg, end)


def test_region_run_of_a_target_without_records(files):
    fa, bam, bam1 = files
    sp = host.bai_region_run(bam1, 1, 0, 3)
    assert sp["empty"] and sp["to_end"]
    assert not host.bai_region_run(bam1, 0, 0, 3)["empty"]
    with pytest.raises(IOError, match="no such target"):
        host.bai_region_run(bam, 5, 0, 1)
    with pytest.raises(IOError, match="no index"):
        host.bai_region_run(bam + ".nope", 0, 0, 1)
