"""File I/O of the host stand-in (indelope_b200/csrc/host/bamio.cpp): a synthetic dataset written as FASTA + BAM and read
back must give the same reads, the same regions of interest and the same oracle VCF; the BAM must be what the
specification says (checked here with Python's gzip on the BGZF members, independent of the C++ reader)."""
import gzip
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from indelope_b200 import build, host
from oracle import pyoracle as orc
import idl_testutil as util

CALL = dict(min_reads=5, min_ctg_len=73, min_event_len=5)


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("io")
    ds = util.small_dataset("pr1", chrom_len=120_000, n_events=24, max_indel=40, n_chroms=2, n_base_rate=0.0005, dup_fraction=0.02)
    fa, bam = str(d / "ref.fa"), str(d / "reads.bam")
    ds.write_fasta(fa)
    ds.write_bam(bam, level=1)
    return ds, fa, bam


def test_bam_is_spec_conformant(files):
    ds, fa, bam = files
    raw = open(bam, "rb").read()
    assert raw[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")  # BGZF EOF marker
    data = gzip.decompress(raw)  # concatenated gzip members
    assert data[:4] == b"BAM\x01"
    l_text, = struct.unpack_from("<i", data, 4)
    text = data[8:8 + l_text].decode()
    assert text.startswith("@HD\tVN:1.6\tSO:coordinate") and "@SQ\tSN:chrS1\tLN:120000" in text
    at = 8 + l_text
    n_ref, = struct.unpack_from("<i", data, at); at += 4
    assert n_ref == 2
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", data, at); at += 4 + l_name + 4
    rois = ds.sweep(min_reads=5)  # keep the owner alive: arrays() are views
    a = rois.arrays()
    n = 0
    while at < len(data):
        block, ref_id, pos, l_name, mapq, _bin, n_cig, flag, l_seq = struct.unpack_from("<iiiBBHHHi", data, at)
        assert pos == a["start"][n] and mapq == a["mapq"][n] and flag == a["flag"][n] and l_seq == a["len"][n]
        at += 4 + block; n += 1
    assert n == len(a["start"])


def test_fasta_and_fai(files):
    ds, fa, bam = files
    lines = open(fa).read().split("\n")
    assert lines[0] == ">chrS1" and all(len(l) <= 60 for l in lines)
    fai = [l.split("\t") for l in open(fa + ".fai").read().strip().split("\n")]
    assert [f[0] for f in fai] == ["chrS1", "chrS2"] and fai[0][1] == "120000" and fai[0][3:] == ["60", "61"]
    txt = open(fa, "rb").read()
    off = int(fai[1][2])
    assert txt[off - 7:off] == b">chrS2\n"


def test_round_trip_gives_identical_regions_and_oracle_vcf(files):
    ds, fa, bam = files
    back = host.Dataset.load(fa, bam, threads=3)
    ra, rb = ds.sweep(min_reads=5), back.sweep(min_reads=5)  # keep the owners alive: arrays() are views
    a, b = ra.arrays(), rb.arrays()
    for k in ("start", "stop", "mapq", "flag", "len", "roi_chrom", "roi_start", "roi_stop", "roi_read_begin", "roi_n_reads", "read_idx"):
        assert np.array_equal(a[k], b[k]), k

    def gather(x, key):  # per-read strings in read order (the generator's pool is in creation order, the file's in file order)
        idx = np.concatenate([np.arange(o, o + l) for o, l in zip(x["seq_off"], x["len"])])
        return x[key][idx]
    assert np.array_equal(gather(a, "bases"), gather(b, "bases")) and np.array_equal(gather(a, "quals"), gather(b, "quals"))
    assert a["chrom_names"] == b["chrom_names"] and all(np.array_equal(x, y) for x, y in zip(a["chrom_seqs"], b["chrom_seqs"]))
    assert len(a["roi_start"]) > 10
    _, v1, _ = orc.call(a, dump_level=0, **CALL)
    _, v2, _ = orc.call(b, dump_level=0, **CALL)
    assert v1 == v2 and v1.count("\n") > 3


def _flatten(groups):
    """regions of a list of groups as (chrom, start, stop, [(read start, stop, mapq, flag, bases, quals), ...])"""
    out = []
    for g in groups:
        a = g.arrays()
        for k in range(len(a["roi_start"])):
            reads = []
            for i in a["read_idx"][a["roi_read_begin"][k]:a["roi_read_begin"][k] + a["roi_n_reads"][k]]:
                o, l = int(a["seq_off"][i]), int(a["len"][i])
                reads.append((int(a["start"][i]), int(a["stop"][i]), int(a["mapq"][i]), int(a["flag"][i]), a["bases"][o:o + l].tobytes(), a["quals"][o:o + l].tobytes()))
            out.append((int(a["roi_chrom"][k]), int(a["roi_start"][k]), int(a["roi_stop"][k]), reads))
    return out


@pytest.mark.parametrize("target_reads", [1, 300, 10**9])
def test_streaming_sweep_equals_the_whole_file_sweep(files, target_reads):
    """idlh_stream_* (incremental gen_roi, bounded memory) against idlh_load + idlh_sweep: same regions, same reads, same order,
    whatever the group size; and the oracle VCF over the concatenated groups is the whole-file one"""
    ds, fa, bam = files
    whole = ds.sweep(min_reads=5)
    st = host.Stream(fa, bam, threads=2, min_reads=5)
    groups = list(st.groups(target_reads))
    assert _flatten(groups) == _flatten([whole])
    assert sum(g.n_rois for g in groups) == whole.n_rois and st.counts() == (ds.n_reads, whole.n_rois)
    if target_reads == 1:
        assert len(groups) >= whole.n_rois // 2  # a group ends at the first record after its target is met
    assert st.targets().header() == whole.header()


def test_streaming_sweep_dense_coverage_without_gaps(tmp_path):
    """whole-contig 40x coverage: one coverage-gap chunk per contig, so every region is found by the incremental scan while
    records are still arriving and cached records are dropped early; decoy contig names are skipped (:41-42)"""
    ds = util.small_dataset("pr1", chrom_len=60_000, n_events=30, max_indel=25, n_chroms=2, coverage=40.0, low_mapq_fraction=0.1, dup_fraction=0.05)
    fa, bam = str(tmp_path / "d.fa"), str(tmp_path / "d.bam")
    ds.write_fasta(fa); ds.write_bam(bam, level=1)
    whole = ds.sweep(min_reads=3)
    assert whole.n_rois > 20
    for tr in (1, 5000):
        assert _flatten(list(host.Stream(fa, bam, min_reads=3).groups(tr))) == _flatten([whole])


def test_reader_rejects_bad_input(files, tmp_path):
    ds, fa, bam = files
    with pytest.raises(IOError, match="cannot open"):
        host.Dataset.load(fa, str(tmp_path / "missing.bam"))
    bad = tmp_path / "bad.bam"
    bad.write_bytes(b"not a bam")
    with pytest.raises(IOError):
        host.Dataset.load(fa, str(bad))
    raw = bytearray(open(bam, "rb").read())
    raw[200] ^= 0xff  # corrupt the first block: inflate error or CRC mismatch
    (tmp_path / "corrupt.bam").write_bytes(bytes(raw))
    with pytest.raises(IOError):
        host.Dataset.load(fa, str(tmp_path / "corrupt.bam"))
    fa2 = tmp_path / "short.fa"
    fa2.write_text(">chrS1\nACGT\n>chrS2\nACGT\n")
    with pytest.raises(IOError, match="different length"):
        host.Dataset.load(str(fa2), bam)
    with pytest.raises(IOError, match="different length"):
        host.Stream(str(fa2), bam)
    with pytest.raises(IOError):
        host.Stream(fa, str(bad))
    with pytest.raises(IOError):
        list(host.Stream(fa, str(tmp_path / "corrupt.bam")).groups())
    cut = tmp_path / "cut.bam"
    cut.write_bytes(bytes(open(bam, "rb").read()[:40000]))  # ends inside a BGZF block
    with pytest.raises(IOError):
        list(host.Stream(fa, str(cut)).groups())


def test_cli_help_and_no_cpu_path(files):
    ds, fa, bam = files
    exe = build.build_cli()
    out = subprocess.run([exe, "--help"], capture_output=True, text=True)
    assert out.returncode == 0 and "--min-event-len" in out.stdout and "--min-reads" in out.stdout and "--threads" in out.stdout
    assert subprocess.run([exe, fa], capture_output=True).returncode == 1
    if not util.has_gpu():
        # every front end fails loudly and prints nothing: streamed, the whole file on the device, target by target, regions
        for args, env in (([], {}), (["-g"], {}), (["-g"], {"INDELOPE_BY_TARGET": "1"}), (["-r", "chrS1"], {})):
            r = subprocess.run([exe, "--min-event-len", "5", "--min-reads", "5"] + args + [fa, bam], capture_output=True, text=True, env=dict(os.environ, **env))
            assert r.returncode == 1 and "no CPU path" in r.stderr and r.stdout == "", (args, env, r.stderr)


def test_cli_by_target_without_index_fails_before_any_output(files, tmp_path):
    """target-by-target decoding needs <bam>.bai: without it the run stops before the header (and before looking for a device)"""
    ds, fa, bam = files
    nobai = tmp_path / "nobai.bam"
    shutil.copy(bam, nobai)
    r = subprocess.run([build.build_cli(), "-g", fa, str(nobai)], capture_output=True, text=True, env=dict(os.environ, INDELOPE_BY_TARGET="1"))
    assert r.returncode == 1 and "no index" in r.stderr and r.stdout == "", r.stderr


@pytest.mark.gpu
def test_cli_vcf_is_byte_identical_to_the_oracle(files):
    """`indelope --min-event-len 5 --min-reads 5 ref.fa reads.bam` (BASELINE.json configs[0] command line) on real files"""
    ds, fa, bam = files
    exe = build.build_cli()
    r = subprocess.run([exe, "--min-event-len", "5", "--min-reads", "5", "-t", "2", fa, bam], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rois = ds.sweep(min_reads=5)
    _, ovcf, cnt = orc.call(rois.arrays(), dump_level=0, **CALL)
    assert r.stdout == rois.header() + ovcf
    assert cnt["variants"] >= 3


@pytest.mark.gpu
def test_cli_gpu_decode_gives_the_same_vcf(files):
    """`indelope --gpu-decode`: BGZF inflate, record parse (idl_bam_open) and gen_roi (idl_bam_sweep, src/indelope.nim:515-545) on the GPU instead of the
    host reader and sweep; same bytes"""
    ds, fa, bam = files
    exe = build.build_cli()
    r = subprocess.run([exe, "--gpu-decode", "--min-event-len", "5", "--min-reads", "5", "-t", "2", fa, bam], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rois = ds.sweep(min_reads=5)
    _, ovcf, cnt = orc.call(rois.arrays(), dump_level=0, **CALL)
    assert r.stdout == rois.header() + ovcf
    # ... and target by target through the index (what the binary does by itself for a file that does not fit in device memory)
    r = subprocess.run([exe, "--gpu-decode", "--min-event-len", "5", "--min-reads", "5", fa, bam], capture_output=True, text=True, env=dict(os.environ, INDELOPE_BY_TARGET="1"))
    assert r.returncode == 0, r.stderr
    assert r.stdout == rois.header() + ovcf


@pytest.mark.gpu
def test_api_call_bam_equals_the_cli_and_the_oracle(files):
    """api.call_bam: the in-process twin of `indelope --gpu-decode` (several small batches in flight)"""
    from indelope_b200 import api
    ds, fa, bam = files
    rois = ds.sweep(min_reads=5)
    _, ovcf, cnt = orc.call(rois.arrays(), dump_level=0, **CALL)
    assert api.call_bam(fa, bam, max_reads=3000, **CALL) == rois.header() + ovcf
    # target by target through the index: every target decoded from its own run of BGZF members (idl_bam_open_slice)
    assert api.call_bam(fa, bam, max_reads=3000, by_target=True, **CALL) == rois.header() + ovcf


@pytest.mark.gpu
def test_one_target_from_its_slice_equals_the_whole_file(files):
    """idl_bam_open_slice: records, per-target range and regions of target c decoded from the members the index points to == the same from the whole file"""
    from indelope_b200 import cuda
    ds, fa, bam = files
    raw = open(bam, "rb").read()
    whole = cuda.Bam(raw)
    W = whole.fetch()
    for c in range(whole.n_ref):
        sp = host.bai_target_span(bam, c)
        b = cuda.Bam(raw[sp["file_begin"]:sp["file_end"]], slice=dict(ref_names=whole.ref_names, ref_len=whole.ref_len, first_record=sp["first_record"],
                                                                     end_member=sp["end_member"], end_offset=sp["end_offset"]))
        lo, hi = b.ref_first[c], b.ref_first[c + 1]
        wlo, whi = whole.ref_first[c], whole.ref_first[c + 1]
        assert hi - lo == whi - wlo > 1000 and lo == 0 and b.n_records == hi   # the chain starts at the target's first record and ends behind its last
        S = b.fetch()
        for k in ("chrom", "start", "stop", "len", "mapq", "flag"):
            assert np.array_equal(S[k][lo:hi], W[k][wlo:whi]), k
        assert np.array_equal(S["bases"][S["seq_off"][lo]:S["seq_off"][hi]], W["bases"][W["seq_off"][wlo]:W["seq_off"][whi]])
        assert np.array_equal(S["cigar"][int(S["cig_off"][lo]):int(S["cig_off"][hi])], W["cigar"][int(W["cig_off"][wlo]):int(W["cig_off"][whi])])
        s1, s2 = b.sweep(c, min_read_coverage=5), whole.sweep(c, min_read_coverage=5)
        for k in ("roi_start", "roi_end", "roi_n_reads"):
            assert np.array_equal(s1[k], s2[k]), k
        assert np.array_equal(s1["read_idx"] - lo, s2["read_idx"] - wlo)
        b.close()
    whole.close()
    with pytest.raises(cuda.IdlError, match="truncated BAM record|malformed|first record|not coordinate sorted|follow records"):
        sp = host.bai_target_span(bam, 1)
        cuda.Bam(raw[sp["file_begin"]:sp["file_end"]], slice=dict(ref_names=["a", "b"], ref_len=[120_000, 120_000], first_record=sp["first_record"] + 3,
                                                                 end_member=sp["end_member"], end_offset=sp["end_offset"]))


def _records_of(data, at, end):
    """(ref_id, pos) of the records in data[at:end] (an uncompressed BAM record stream)"""
    out = []
    while at < end:
        bs, ref_id, pos = struct.unpack_from("<iii", data, at)
        out.append((ref_id, pos)); at += 4 + bs
    assert at == end
    return out


def test_target_span_from_the_index(files):
    """idlh_bai_target_span: the run of BGZF members that holds one target's records and where its record chain starts and ends inside it -- checked by
    inflating exactly that run with gzip and walking the records"""
    ds, fa, bam = files
    raw = open(bam, "rb").read()
    whole = gzip.decompress(raw)
    l_text, = struct.unpack_from("<i", whole, 4); at = 8 + l_text
    n_ref, = struct.unpack_from("<i", whole, at); at += 4
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", whole, at); at += 4 + l_name + 4
    allrec = _records_of(whole, at, len(whole))
    for c in range(2):
        sp = host.bai_target_span(bam, c)
        assert sp is not None and 0 <= sp["file_begin"] < sp["file_end"] <= len(raw)
        run = raw[sp["file_begin"]:sp["file_end"]]
        inflated = gzip.decompress(run)                                  # whole members: decompresses cleanly
        # where the chain ends: the inflated size of the members in front of end_member + end_offset
        end = len(gzip.decompress(run[:sp["end_member"]])) + sp["end_offset"] if sp["end_member"] else sp["end_offset"]
        recs = _records_of(inflated, sp["first_record"], end)
        assert recs == [r for r in allrec if r[0] == c] and len(recs) > 1000
    with pytest.raises(IOError):
        host.bai_target_span(bam, 7)
    with pytest.raises(IOError):
        host.bai_target_span(bam + ".nope", 0)


def test_targets_from_the_header_alone(files, tmp_path):
    """idlh_load_targets: the FASTA's sequences in the BAM header's order; of the BAM only the header members are read"""
    import ctypes as C
    ds, fa, bam = files
    L = host.lib()
    L.idlh_load_targets.restype = C.c_void_p
    L.idlh_load_targets.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]
    err = C.create_string_buffer(512)
    h = L.idlh_load_targets(fa.encode(), bam.encode(), err, 512)
    assert h, err.value
    d = host.Dataset(_handle=h)
    names, seqs = d.sequences()
    assert names == ["chrS1", "chrS2"] and d.n_reads == 0 and len(seqs[1]) == 120_000
    cut = tmp_path / "head.bam"
    cut.write_bytes(open(bam, "rb").read()[:70_000])          # the header survives a file cut off behind its first members
    h2 = L.idlh_load_targets(fa.encode(), str(cut).encode(), err, 512)
    assert h2
    host.Dataset(_handle=h2)
    assert not L.idlh_load_targets(fa.encode(), fa.encode(), err, 512) and b"not a BAM" in err.value


def test_fasta_only_dataset_and_target_order(files, tmp_path):
    """idlh_load_fasta + idlh_dataset_set_targets: what the device path keeps of the host reader -- the sequences, ordered as the BAM header lists them"""
    ds, fa, bam = files
    ref = host.Dataset.load_fasta(fa)
    names, seqs = ref.sequences()
    assert names == ["chrS1", "chrS2"] and [len(s) for s in seqs] == [120_000, 120_000]
    second = bytes(seqs[1][:50])   # (the views die with the reordering)
    ref.set_targets(["chrS2", "chrS1"], [120_000, 120_000])
    n2, s2 = ref.sequences()
    assert n2 == ["chrS2", "chrS1"] and bytes(s2[0][:50]) == second
    with pytest.raises(IOError, match="not in the FASTA"):
        host.Dataset.load_fasta(fa).set_targets(["chrX"], [10])
    with pytest.raises(IOError, match="different length"):
        host.Dataset.load_fasta(fa).set_targets(["chrS1"], [5])
    with pytest.raises(IOError):
        host.Dataset.load_fasta(str(tmp_path / "missing.fa"))


def _parse_bai(path):
    """the index as the SAM specification lays it out (5.2), read with struct alone"""
    b = open(path, "rb").read()
    assert b[:4] == b"BAI\x01"
    n_ref, = struct.unpack_from("<i", b, 4); at = 8
    refs = []
    for _ in range(n_ref):
        n_bin, = struct.unpack_from("<i", b, at); at += 4
        bins = {}
        for _ in range(n_bin):
            bn, n_chunk = struct.unpack_from("<Ii", b, at); at += 8
            bins[bn] = [struct.unpack_from("<QQ", b, at + 16 * c) for c in range(n_chunk)]; at += 16 * n_chunk
        n_intv, = struct.unpack_from("<i", b, at); at += 4
        lin = list(struct.unpack_from("<%dQ" % n_intv, b, at)); at += 8 * n_intv
        refs.append((bins, lin))
    assert at == len(b)
    return refs


def _reg2bin(beg, end):
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def test_bai_index_is_spec_conformant(files):
    """the .bai written next to the BAM (the reference opens its BAM with index=true, src/indelope.nim:595): every record lies inside a
    chunk of its bin, chunks are ordered and start at record boundaries, the linear index holds the first record of each 16 kb window"""
    ds, fa, bam = files
    refs = _parse_bai(bam + ".bai")
    assert len(refs) == 2
    rois = ds.sweep(min_reads=5)
    a = rois.arrays()
    # virtual offsets of every record, recomputed from the BGZF members with gzip/zlib alone
    raw = open(bam, "rb").read()
    blocks, at, uoff = [], 0, 0
    while at < len(raw):
        bsize = struct.unpack_from("<H", raw, at + 16)[0] + 1
        isize, = struct.unpack_from("<I", raw, at + bsize - 4)
        blocks.append((at, uoff, isize)); uoff += isize; at += bsize
    data = gzip.decompress(raw)
    def voff(u):
        k = max(i for i, bl in enumerate(blocks) if bl[1] <= u and (bl[2] > 0 or bl[1] < u))
        while blocks[k][2] == 0 or u - blocks[k][1] >= blocks[k][2]:
            k += 1
        return blocks[k][0] << 16 | (u - blocks[k][1])
    l_text, = struct.unpack_from("<i", data, 4); at = 8 + l_text
    n_ref, = struct.unpack_from("<i", data, at); at += 4
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", data, at); at += 4 + l_name + 4
    n = 0
    first_in_window = [dict(), dict()]
    while at < len(data):
        block, ref_id, pos = struct.unpack_from("<iii", data, at)
        v0 = voff(at)
        stop = int(a["stop"][n])
        bins, lin = refs[ref_id]
        chunks = bins[_reg2bin(pos, max(stop, pos + 1))]
        assert any(c0 <= v0 < c1 for c0, c1 in chunks)
        for w in range(pos >> 14, ((max(stop, pos + 1) - 1) >> 14) + 1):
            first_in_window[ref_id].setdefault(w, v0)
        at += 4 + block; n += 1
    for r in range(2):
        bins, lin = refs[r]
        for ch in bins.values():
            assert all(c0 < c1 for c0, c1 in ch) and all(ch[i][1] <= ch[i + 1][0] for i in range(len(ch) - 1))
        for w, v in first_in_window[r].items():
            assert lin[w] == v


def test_region_queries_through_the_index(files):
    """idlh_load_region = b.querys("chr:beg-end") (src/indelope.nim:454-459,527): the records that overlap the interval, in file order,
    found through the .bai; the whole-target query feeds the sweep exactly like the sequential read"""
    ds, fa, bam = files
    full = host.Dataset.load(fa, bam, threads=2)
    rf = full.sweep(min_reads=5); af = rf.arrays()
    n0 = int((np.array([full.chrom_reads(0)["first_read"], full.chrom_reads(1)["first_read"]])[1]))
    rng = np.random.default_rng(4)
    queries = [("chrS1", 0, 0), ("chrS2", 0, 0), ("chrS1", 50_000, 50_001), ("chrS2", 119_000, 0), ("chrS1", 16_383, 16_385), ("chrS2", 0, 10)]
    queries += [("chrS%d" % (1 + int(rng.integers(0, 2))), int(b), int(b + rng.integers(1, 40_000))) for b in rng.integers(0, 119_000, 12)]
    for name, beg, end in queries:
        c = int(name[-1]) - 1
        sub = host.Dataset.load_region(fa, bam, name, beg, end)
        cr = full.chrom_reads(c)
        e = end if end > 0 else cr["chrom_len"]
        want = np.nonzero((cr["start"] < e) & (cr["stop"] > beg))[0]
        got = sub.chrom_reads(c)
        assert len(got["start"]) == len(want), (name, beg, end)
        assert np.array_equal(got["start"], cr["start"][want]) and np.array_equal(got["stop"], cr["stop"][want]) and np.array_equal(got["flag"], cr["flag"][want])
        assert np.array_equal(got["cigar"], np.concatenate([cr["cigar"][int(cr["cig_off"][i]):int(cr["cig_off"][i + 1])] for i in want]) if len(want) else np.zeros(0, np.uint32))
    # per-target queries give the regions of the sequential sweep (what `for target in targets: b.querys(target.name)` relies on)
    for c, name in enumerate(("chrS1", "chrS2")):
        sub = host.Dataset.load_region(fa, bam, name)
        rs = sub.sweep(min_reads=5); a = rs.arrays()
        sel = af["roi_chrom"] == c
        assert np.array_equal(a["roi_start"][a["roi_chrom"] == c], af["roi_start"][sel]) and np.array_equal(a["roi_n_reads"][a["roi_chrom"] == c], af["roi_n_reads"][sel])
    with pytest.raises(IOError):
        host.Dataset.load_region(fa, bam, "chrNope")
