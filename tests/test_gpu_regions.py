"""`indelope -r / -R` and api.call_bam(regions=, bed=) against the oracle, and idl_bam_sweep_window against the whole target's idl_bam_sweep.

The output for a set of intervals is defined as the VCF header + the oracle's records for the whole-file run's regions of interest that overlap an
interval (roi_start < end and roi_end >= beg), called in the whole-file order with the dedup applied over that subsequence.  The slices of the file the
command line decodes, the zones it sweeps and the retries it makes (DESIGN.md 4a) must not change a byte of that."""
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from indelope_b200 import api, build, cuda, host
from oracle import pyoracle as orc
import idl_testutil as util

pytestmark = pytest.mark.gpu

CALL = dict(min_reads=5, min_ctg_len=73, min_event_len=5)
SWEEP = dict(min_event_support=3, min_read_coverage=5, max_read_coverage=600)


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """the test_files dataset with two ~400 kb targets: 25 linear-index windows each"""
    d = tmp_path_factory.mktemp("regions")
    ds = util.small_dataset("pr1", chrom_len=400_000, n_events=60, max_indel=40, n_chroms=2, n_base_rate=0.0005, dup_fraction=0.02)
    fa, bam = str(d / "ref.fa"), str(d / "reads.bam")
    ds.write_fasta(fa)
    ds.write_bam(bam, level=1)
    rois = ds.sweep(min_reads=5)
    return ds, fa, bam, rois, rois.arrays(), d


def expected(rois, arrays, per_target, call=CALL):
    """header + the oracle's records of the whole-file regions that overlap an interval; per_target = {target: [(beg, end), ...]} (0-based, half open)"""
    keep = []
    rc, rs, re_ = np.asarray(arrays["roi_chrom"]), np.asarray(arrays["roi_start"]), np.asarray(arrays["roi_stop"])
    for k in range(len(rs)):
        if any(rs[k] < e and re_[k] >= b for b, e in per_target.get(int(rc[k]), ())):
            keep.append(k)
    if not keep:
        return rois.header(), 0
    _, ovcf, _ = orc.call(util.region_subset(arrays, keep), dump_level=0, **call)
    return rois.header() + ovcf, len(keep)


def run_cli(fa, bam, args, call=CALL, env=None):
    exe = build.build_cli()
    opts = ["--min-reads", str(call["min_reads"]), "--min-contig-len", str(call["min_ctg_len"]), "--min-event-len", str(call["min_event_len"])]
    return subprocess.run([exe] + opts + args + [fa, bam], capture_output=True, text=True, env=dict(os.environ, INDELOPE_TIMING="1", **(env or {})))


def timing(stderr, what):
    m = re.search(r"indelope timing \(regions\):.* %s (\d+)" % what, stderr.replace(",", ""))
    assert m, stderr
    return int(m.group(1))


# ---- idl_bam_sweep_window ---------------------------------------------------------------------------------------------------------------------------

def window_model(ev, cut, zlo, zhi, min_ev):
    """runs of the zone [zlo, zhi] as the device forms them from the whole target's evidence and cuts (positions outside the zone do not exist)"""
    p = np.arange(zlo, zhi + 1)
    f = ev[zlo:zhi + 1] >= min_ev
    prev = np.concatenate([[False], f[:-1]])
    nxt = np.concatenate([f[1:], [False]])
    c_here = cut[zlo:zhi + 1].astype(bool)
    c_next = np.concatenate([cut[zlo + 1:zhi + 1].astype(bool), [False]])
    starts = p[f & (~prev | c_here)]
    ends = p[f & (~nxt | c_next)]
    assert len(starts) == len(ends)
    return starts, ends


def overlaps(rs, re_, ivs):
    return any(rs < e and re_ >= b for b, e in ivs)


def test_sweep_window_equals_the_whole_target(files):
    """~200 random zones and interval sets on the whole-file resident BAM: the regions returned are the whole target's regions that overlap an interval and
    lie strictly inside the zone (same records, same order), and n_edge counts the selected runs that touch an inner edge"""
    ds, fa, bam, rois, arrays, d = files
    b = cuda.Bam(open(bam, "rb").read())
    rng = random.Random(404)
    n_checked = n_edges = 0
    for c in range(b.n_ref):
        L = b.ref_len[c]
        whole = b.sweep(c, evidence=True, **SWEEP)
        ev = whole["evidence"]
        recs = b.fetch(np.arange(b.ref_first[c], b.ref_first[c + 1]), what=0)
        skip = (recs["flag"].astype(np.int64) & (0x400 | 0x200 | 0x4 | 0x800 | 0x100)) != 0
        stopv = np.where(skip, np.iinfo(np.int64).min, recs["stop"].astype(np.int64))
        before = np.concatenate([[np.iinfo(np.int64).min], np.maximum.accumulate(stopv)[:-1]])
        cut = np.zeros(L + 2, np.uint8)
        s = recs["start"].astype(np.int64)
        cs = s[(s > before) & (s >= 0) & (s <= L)]
        cut[cs] = 1
        rbeg = np.concatenate([whole["roi_read_begin"], [len(whole["read_idx"])]])
        zones = [(0, L), (0, 0), (L, L), (0, 5000), (L - 5000, L), (17, 17), (16_384, 32_768)]
        zones += [tuple(sorted(rng.randrange(0, L + 1) for _ in range(2))) for _ in range(63)]
        # zones with an edge inside a region, or on its first or last base, and an interval over that region: the edge counts
        n_fixed = len(zones)
        for _ in range(30):
            k = rng.randrange(len(whole["roi_start"]))
            p = rng.choice([int(whole["roi_start"][k]), int(whole["roi_end"][k]), (int(whole["roi_start"][k]) + int(whole["roi_end"][k])) // 2])
            other = rng.randrange(0, L + 1)
            zones.append((min(p, other), max(p, other)))
        for zi, (zlo, zhi) in enumerate(zones):
            n_iv = 0 if zi == 3 else rng.choice([1, 1, 2, 3, 10])
            pts = sorted(rng.randrange(0, L) for _ in range(2 * n_iv))
            ivs = [(pts[2 * k], pts[2 * k + 1] + 1) for k in range(n_iv)]
            if zi >= n_fixed:
                ivs = [(max(0, zlo - 100), min(L, zlo + 100)), (max(0, zhi - 100), min(L, zhi + 100))]
            ivs = [iv for k, iv in enumerate(ivs) if k == 0 or iv[0] >= ivs[k - 1][1]]
            if zi == 0:
                ivs = [(0, L)]
            got = b.sweep_window(c, zlo, zhi, [x[0] for x in ivs], [x[1] for x in ivs], evidence=True, **SWEEP)
            assert np.array_equal(got["evidence"], ev[zlo:zhi + 1])
            want = [k for k in range(len(whole["roi_start"]))
                    if overlaps(whole["roi_start"][k], whole["roi_end"][k], ivs) and (whole["roi_start"][k] > zlo or zlo == 0) and whole["roi_start"][k] >= zlo
                    and (whole["roi_end"][k] < zhi or zhi == L) and whole["roi_end"][k] <= zhi]
            assert list(got["roi_start"]) == [whole["roi_start"][k] for k in want], (c, zlo, zhi, ivs)
            assert list(got["roi_end"]) == [whole["roi_end"][k] for k in want]
            assert list(got["roi_n_reads"]) == [whole["roi_n_reads"][k] for k in want]
            idx = [whole["read_idx"][rbeg[k]:rbeg[k + 1]] for k in want]
            assert np.array_equal(got["read_idx"], np.concatenate(idx) if idx else np.zeros(0, np.int64))
            ws, we = window_model(ev, cut, zlo, zhi, SWEEP["min_event_support"])
            sel = [overlaps(x, y, ivs) for x, y in zip(ws, we)]
            e_lo = sum(1 for x, y, t in zip(ws, we, sel) if t and zlo > 0 and x == zlo)
            e_hi = sum(1 for x, y, t in zip(ws, we, sel) if t and zhi < L and y == zhi)
            assert got["n_edge"] == (e_lo, e_hi), (c, zlo, zhi, ivs)
            assert got["n_runs"] == len(ws)
            n_checked += len(want); n_edges += e_lo + e_hi
        # the whole target through the window entry point with one interval over everything is idl_bam_sweep
        full = b.sweep_window(c, 0, L, [0], [L], **SWEEP)
        for k in ("roi_start", "roi_end", "roi_n_reads", "read_idx"):
            assert np.array_equal(full[k], whole[k]), k
    assert n_checked > 200 and n_edges > 5
    with pytest.raises(cuda.IdlError):
        b.sweep_window(0, 10, 5, [0], [1])                 # zone_hi < zone_lo
    with pytest.raises(cuda.IdlError):
        b.sweep_window(0, 0, b.ref_len[0] + 1, [0], [1])   # past the target
    with pytest.raises(cuda.IdlError):
        b.sweep_window(0, 0, 100, [5, 3], [6, 4])          # unsorted intervals
    b.close()


# ---- the command line and api.call_bam ---------------------------------------------------------------------------------------------------------------

def bed_of(path, lines):
    with open(path, "w") as f:
        f.write("".join("%s\t%d\t%d\n" % x for x in lines))
    return str(path)


def test_regions_through_the_command_line_and_the_api(files):
    ds, fa, bam, rois, arrays, d = files
    names = ["chrS1", "chrS2"]
    L = 400_000
    rs, re_, rc = np.asarray(arrays["roi_start"]), np.asarray(arrays["roi_stop"]), np.asarray(arrays["roi_chrom"])
    k = int(np.argmax((rc == 0) & (re_ - rs >= 2)))                     # a region of a few bases on the first target
    a0, a1 = int(rs[k]), int(re_[k])
    cases = [  # (-r strings, BED lines, {target: intervals})
        (["chrS1:200,001-210,000"], [], {0: [(200_000, 210_000)]}),
        (["chrS1:1-1"], [], {0: [(0, 1)]}),
        (["chrS2:400000-400000"], [], {1: [(L - 1, L)]}),
        (["chrS1:%d-%d" % (a0 + 2, a0 + 2)], [], {0: [(a0 + 1, a0 + 2)]}),             # inside a region
        (["chrS1:%d-%d" % (a0 - 5, a0)], [], {0: [(a0 - 6, a0)]}),                     # ends one base before it
        (["chrS1:%d-%d" % (a1 + 2, a1 + 9)], [], {0: [(a1 + 1, a1 + 9)]}),             # starts one base after it
        ([], [("chrS1", a0 - 6, a0)], {0: [(a0 - 6, a0)]}),                            # the same in BED coordinates
        ([], [("chrS1", a0 - 6, a0 + 1)], {0: [(a0 - 6, a0 + 1)]}),
        ([], [("chrS1", a1 + 1, a1 + 9)], {0: [(a1 + 1, a1 + 9)]}),
        ([], [("chrS1", a1, a1 + 9)], {0: [(a1, a1 + 9)]}),
        ([], [("chrS2", 5000, 9000), ("chrS2", 100_000, 190_000), ("chrS2", 5000, 9000), ("chrS2", 8000, 30_000), ("chrS1", 0, 16_384)],
         {0: [(0, 16_384)], 1: [(5000, 30_000), (100_000, 190_000)]}),               # duplicate, overlapping, out of order
        (["chrS2:300000-350000", "chrS1:1000-2000"], [], {0: [(999, 2000)], 1: [(299_999, 350_000)]}),   # two targets in reverse header order
        (["chrS1"], [("chrS2", 16_384, 32_768)], {0: [(0, L)], 1: [(16_384, 32_768)]}),
    ]
    # an interval without any region: header only
    gaps = [(int(re_[j]) + 1, int(rs[j + 1])) for j in range(len(rs) - 1) if rc[j] == rc[j + 1] == 0 and rs[j + 1] - re_[j] > 3000]
    cases.append(([], [("chrS1", gaps[0][0] + 1000, gaps[0][0] + 1010)], {0: [(gaps[0][0] + 1000, gaps[0][0] + 1010)]}))
    rng = random.Random(7)
    for _ in range(20):
        lines = []
        for _ in range(10):
            c = rng.randrange(2); b0 = rng.randrange(0, L); lines.append((names[c], b0, min(L, b0 + rng.choice([1, 50, 500, 5000, 40_000]))))
        per = {}
        for n, b0, e0 in lines:
            per.setdefault(names.index(n), []).append((b0, e0))
        cases.append(([], lines, per))
    n_empty = 0
    for i, (rstr, lines, per) in enumerate(cases):
        want, n = expected(rois, arrays, per)
        n_empty += n == 0
        args = []
        for r in rstr:
            args += ["-r", r]
        bed = bed_of(d / ("c%d.bed" % i), lines) if lines else None
        if bed:
            args += ["-R", bed]
        r = run_cli(fa, bam, args)
        assert r.returncode == 0, r.stderr
        assert r.stdout == want, (i, rstr, lines, util.diff_lines(want, r.stdout))
        assert timing(r.stderr, "regions") == n
        if i % 4 == 0:
            assert api.call_bam(fa, bam, regions=rstr or None, bed=bed, max_reads=3000, **CALL) == want, (i, rstr, lines)
    assert n_empty >= 1
    # with --gpu-decode the same path is taken
    r = run_cli(fa, bam, ["-g", "-r", "chrS1:200,001-210,000"])
    assert r.returncode == 0 and r.stdout == expected(rois, arrays, {0: [(200_000, 210_000)]})[0]


def test_errors_leave_stdout_empty(files, tmp_path):
    ds, fa, bam, rois, arrays, d = files
    nobai = tmp_path / "nobai.bam"
    shutil.copy(bam, nobai)
    bad = tmp_path / "bad.bed"
    bad.write_text("chrS1\t10\t20\nchrS1\t30\tx\n")
    for args, path, msg in ((["-r", "chrS1:1-100"], str(nobai), "no index"), (["-r", "chrQ:1-100"], bam, "no such target"),
                            (["-R", str(bad)], bam, "line 2"), (["-r", "chrS1:0-5"], bam, "beg must be")):
        r = run_cli(fa, path, args)
        assert r.returncode == 1 and r.stdout == "" and msg in r.stderr, (args, r.stderr)
    with pytest.raises(ValueError, match="no such target"):
        api.call_bam(fa, bam, regions=["chrQ:1-5"])
    with pytest.raises(IOError, match="no index"):
        api.call_bam(fa, str(nobai), regions=["chrS1:1-5"])
    with pytest.raises(IOError, match="no index"):
        api.call_bam(fa, str(nobai), by_target=True)


def test_by_target_is_the_regions_loop_over_whole_targets(files):
    """target-by-target decoding goes through the sliced loop with one interval per target: a whole target is one slice, swept once"""
    ds, fa, bam, rois, arrays, d = files
    want = api.call_bam(fa, bam, **CALL)
    t = []
    assert api.call_bam(fa, bam, by_target=True, timings=t, **CALL) == want
    stats = [x for x in t if "slices" in x]
    assert [x["target"] for x in stats] == [0, 1] and all(x["slices"] == 1 and x["retries"] == 0 for x in stats), stats
    r = run_cli(fa, bam, ["-g"], env={"INDELOPE_BY_TARGET": "1"})
    assert r.returncode == 0 and r.stdout == want, r.stderr
    assert timing(r.stderr, "slices") == 2 and timing(r.stderr, "retries") == 0


# ---- a directed fixture: long evidence runs, slices that must grow, a deep region across a zone edge ---------------------------------------------------

def directed_files(d):
    rng = np.random.default_rng(99)
    L = 200_000
    ref = util.random_seq(rng, L)
    reads = []

    def plain(at, n=150, mapq=60, cigar=None, seq=None):
        reads.append(dict(start=at, seq=seq or ref[at:at + n], cigar=cigar or [("M", n)], mapq=mapq))

    # background coverage every 25 bases, none under the N skips (their region would hold more than 600 reads)
    for at in range(0, L - 150, 25):
        if not 59_000 <= at <= 101_000:
            plain(at)
    # (1) a 1.5 kb deletion carried by 6 reads, its evidence from 48 452 to 49 952: across the window edge 49 152
    D, DL = 48_452, 1500
    for k in range(6):
        a = 40 + 12 * k
        reads.append(dict(start=D - a, seq=ref[D - a:D] + ref[D + DL:D + DL + 150 - a], cigar=[("M", a), ("D", DL), ("M", 150 - a)], mapq=60))
    # (2) 5 reads with a 40 kb N skip, from 60 000 to 100 000: four 16 kb windows of evidence, starting before any zone around 80 000
    for k in range(5):
        s = 60_000 - 40 + 7 * k
        reads.append(dict(start=s, seq=ref[s:s + 40] + ref[s + 40_040:s + 40_100], cigar=[("M", 40), ("N", 40_000), ("M", 60)], mapq=60))
    # (3) 700 reads with a 3-base deletion at 32 767 (evidence 32 767 .. 32 769, across the window edge 32 768): over the 600-read cap
    for k in range(700):
        a = 20 + (k % 100)
        s = 32_767 - a
        reads.append(dict(start=s, seq=ref[s:32_767] + ref[32_770:32_770 + 150 - a], cigar=[("M", a), ("D", 3), ("M", 150 - a)], mapq=60))
    reads.sort(key=lambda r: r["start"])
    fa, raw_bam, bam = os.path.join(d, "dir.fa"), os.path.join(d, "dir_raw.bam"), os.path.join(d, "dir.bam")
    with open(fa, "w") as f:
        f.write(">chrD\n%s\n" % "\n".join(ref[i:i + 60] for i in range(0, L, 60)))
    recs = [util.bam_record(0, r["start"], r["cigar"], r["seq"], mapq=r["mapq"], name=b"d%d" % k) for k, r in enumerate(reads)]
    with open(raw_bam, "wb") as f:
        f.write(util.bgzf_compress(util.bam_bytes([("chrD", L)], recs)))
    ds = host.Dataset.load(fa, raw_bam)        # the host reader, then its writer: the same records with a .bai
    ds.write_bam(bam, level=1)
    return ds, fa, bam


def test_directed_fixture(tmp_path):
    ds, fa, bam = directed_files(str(tmp_path))
    call = dict(min_reads=3, min_ctg_len=73, min_event_len=4)
    rois = ds.sweep(min_reads=3)
    arrays = rois.arrays()
    rs, re_, nr = np.asarray(arrays["roi_start"]), np.asarray(arrays["roi_stop"]), np.asarray(arrays["roi_n_reads"])
    # the fixture is what it claims: a region longer than the deletion across 49 152, one over the N skips, none kept at 32 768 (over the cap)
    assert any(s < 49_152 <= e and e - s >= 1400 for s, e in zip(rs, re_))
    assert any(s <= 60_100 and e >= 99_900 for s, e in zip(rs, re_))
    assert not any(s <= 32_769 and e >= 32_767 for s, e in zip(rs, re_))
    for rstr, per, retries in ((["chrD:49,200-49,300"], {0: [(49_199, 49_300)]}, 1),     # zone edge 49 153 inside the deletion's region
                               (["chrD:80,001-80,010"], {0: [(80_000, 80_010)]}, 2),     # inside the N skip: grows over several windows on both sides
                               (["chrD:32,770-32,800"], {0: [(32_769, 32_800)]}, 1),     # the deep region touches zone_lo = 32 769
                               (["chrD:32,770-32,800", "chrD:49,200-49,300", "chrD:80,001-80,010", "chrD:150,000-150,100"],
                                {0: [(32_769, 32_800), (49_199, 49_300), (80_000, 80_010), (149_999, 150_100)]}, 2)):   # the first two share a slice
        want, n = expected(rois, arrays, per, call)
        r = run_cli(fa, bam, sum((["-r", x] for x in rstr), []), call)
        assert r.returncode == 0, r.stderr
        assert r.stdout == want, (rstr, util.diff_lines(want, r.stdout))
        assert timing(r.stderr, "retries") >= retries, r.stderr
        t = []
        assert api.call_bam(fa, bam, regions=rstr, timings=t, **call) == want
        assert sum(x.get("retries", 0) for x in t) >= retries
