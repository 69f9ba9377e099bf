"""The calling path at the limits its parameters accept, against the oracle bit for bit: read lengths no dataset reaches (300-2000 bases, trimmed
lengths on the kernels' switch points), MAPQs over 0-255, max_contig_len / max_reads_per_region / n_streams away from their defaults, and the
per-region status bits.  A region that a limit drops is predicted exactly (the oracle's limit lines, dump bit 64); every other region of its batch
equals the oracle's records, and the VCF equals the oracle's over the regions that were kept."""
import os

import numpy as np
import pytest

import idl_testutil as util
from indelope_b200 import abi, api, cuda, host
from oracle import pyoracle as orc
from test_gpu_pipeline import assert_same, run_both
from test_limits_fixtures import LEN_SETS

pytestmark = pytest.mark.gpu

RS_CONTIG_OVERFLOW, RS_CORR_OVERFLOW, RS_DP_OVERFLOW, RS_READ_TOO_LONG, RS_BAD_INPUT = 0, 1, 2, 4, 6  # bit numbers of IDL_RS_*
DIRECTED = dict(min_reads=3, min_ctg_len=73, min_event_len=4)


def _device(arrays, level=31, **kw):
    caller = api.Caller(0, out_flags=abi.OUT_SUPPORT, **kw)
    try:
        vcf, dump = caller.call(host.Rois(arrays=arrays), dump_level=level)
        counts = list(caller.status_counts)
    finally:
        caller.close()
    return vcf, dump, counts


def assert_flagged_exactly(arrays, flagged, bit, capfd, dump, vcf, counts, min_reads, min_ctg_len, min_event_len):
    """regions `flagged` carry status bit `bit` and nothing else; every other region's records equal the oracle's; the VCF equals the oracle's
    over the kept regions; status_counts counts the flagged regions and stderr names them"""
    kw = dict(min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len, use_ref_ksw2=orc.have_ref())
    odump, _, _ = orc.call(arrays, dump_level=31, **kw)
    g, o = util.by_region(dump), util.by_region(odump)
    n = len(arrays["roi_start"])
    for k in range(n):
        if k in flagged:
            assert len(g[k]) == 1 and g[k][0].startswith("R\t") and g[k][0].endswith("\tn=0"), (k, g[k][:3])
        else:
            assert g.get(k) == o.get(k), "region %d:\n%s" % (k, util.diff_lines("\n".join(o.get(k, [])), "\n".join(g.get(k, [])), 4))
    keep = [k for k in range(n) if k not in flagged]
    _, ovcf, _ = orc.call(util.region_subset(arrays, keep), dump_level=0, **kw)
    assert vcf == ovcf
    assert counts[bit] == len(flagged) and sum(counts) == len(flagged), counts
    err = capfd.readouterr().err
    name = {RS_CONTIG_OVERFLOW: "max_contig_len", RS_CORR_OVERFLOW: "voting sites", RS_READ_TOO_LONG: "max_read_len",
            RS_BAD_INPUT: "malformed read record"}[bit]
    assert sum(name in l for l in err.splitlines() if "indelope: warning: region" in l) == min(len(flagged), 20)


# ---- 1. read lengths ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("read_len", [300, 400, 512])
def test_long_reads_at_the_default_parameters(read_len):
    ds = util.small_dataset("pr1", chrom_len=200_000, n_events=40, max_indel=40, read_len=read_len, tr_fraction=0.3, seed=400 + read_len)
    rois = ds.sweep(min_reads=5)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag="len%d" % read_len)
    assert cnt["regions"] > 10 and cnt["dp_b"] > 0
    assert_same(dump, vcf, odump, ovcf)


@pytest.mark.parametrize("n_streams", [2, 1, 8])
def test_trimmed_lengths_on_kernel_boundaries(n_streams):
    """reads of 160 and 161 bases in one AL event (ksw_rows_w switches at 160, per warp); 27/28 (K, K + 1) and lengths = 0, 1, 63 mod 64 for the
    k-mer windows; a generator slice of 300-base reads besides; with one lane and with eight, in batches of about 40 reads"""
    arrays = util.length_fixture(LEN_SETS)
    rois = host.Rois(arrays=arrays)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, arrays, tag="lens_%d" % n_streams, n_streams=n_streams, max_reads=40 if n_streams != 2 else 400_000, **DIRECTED)
    assert cnt["al_events"] >= 2 and cnt["dp_b"] > 0
    assert_same(dump, vcf, odump, ovcf)
    if n_streams != 2:
        ds = util.small_dataset("pr1", chrom_len=120_000, n_events=20, max_indel=40, read_len=300, tr_fraction=0.3, seed=7)
        g = ds.sweep(min_reads=5)
        plans = api.plan_batches(g, 0, g.n_rois, max_reads=40)
        assert len(plans) > 2 * n_streams
        dump, vcf, odump, ovcf, cnt, tm = run_both(g, g.arrays(), tag="lanes_%d" % n_streams, n_streams=n_streams, max_reads=40)
        assert len(tm) == len(plans) and cnt["dp_b"] > 0
        assert_same(dump, vcf, odump, ovcf)


def test_512_called_and_513_dropped(capfd):
    arrays = util.length_fixture([[512] * 6, [512] * 5 + [513], [150] * 8])
    vcf, dump, counts = _device(arrays, **DIRECTED)
    assert_flagged_exactly(arrays, {1}, RS_READ_TOO_LONG, capfd, dump, vcf, counts, **DIRECTED)
    assert vcf.count("\n") == 1


def _free_bytes():
    import ctypes as C
    free, total = C.c_size_t(), C.c_size_t()
    assert cuda.lib().idl_device_memory(0, C.byref(free), C.byref(total)) == 0
    return free.value


def test_960_base_reads_and_the_read_length_limit(capfd):
    """Call-site B stages the trimmed read in shared memory; with the unbanded default that holds 960 bases.  idl_create refuses a larger
    max_read_len, so a longer read drops its region (IDL_RS_READ_TOO_LONG) and never its batch.  At max_read_len = 960: generator reads
    of 960 bases through the AL fallback with one lane (kernel-2 workspaces sized for the groups that fit the lane's budget), bit for bit,
    and a 1000-base read that drops only its own region.  The device memory the context took is written to the output directory (a
    difference of free memory on a shared device: reported, not asserted)"""
    for n, ok in ((960, True), (961, False), (2048, False)):
        if ok:
            cuda.Context(0, abi.default_params(max_read_len=n)).close()
        else:
            with pytest.raises(cuda.IdlError, match="bad argument"):
                cuda.Context(0, abi.default_params(max_read_len=n))
    ds = util.small_dataset("pr1", chrom_len=80_000, n_events=16, max_indel=40, read_len=960, coverage=20.0, tr_fraction=0.8, tr_max_unit=4,
                            seed=960)
    rois = ds.sweep(min_reads=5)
    kw = dict(min_reads=5, min_ctg_len=73, min_event_len=5)
    free0 = _free_bytes()
    caller = api.Caller(0, out_flags=abi.OUT_SUPPORT, max_read_len=960, max_contig_len=8192, n_streams=1, **kw)
    try:
        vcf, dump = caller.call(rois, dump_level=31)
        used = free0 - _free_bytes()
    finally:
        caller.close()
    with open(os.path.join(util.out_dir(), "limits_memory.txt"), "a") as f:
        f.write("read_len 960: %.2f GB of device memory held by the context\n" % (used / 1e9))
    odump, ovcf, cnt = orc.call(rois.arrays(), dump_level=31, use_ref_ksw2=orc.have_ref(), **kw)
    assert cnt["regions"] > 3 and cnt["variants"] > 0 and cnt["dp_a"] > 0 and cnt["dp_b"] > 0
    assert_same(dump, vcf, odump, ovcf)
    arrays = util.length_fixture([[960] * 6, [960] * 5 + [1000], [150] * 8])
    vcf, dump, counts = _device(arrays, max_read_len=960, **DIRECTED)
    assert_flagged_exactly(arrays, {1}, RS_READ_TOO_LONG, capfd, dump, vcf, counts, **DIRECTED)


# ---- 2. MAPQ over 0-255 ---------------------------------------------------------------------------------------------------------------------
def test_mapq_over_its_whole_range():
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=60, max_indel=40, tr_fraction=0.3, seed=81)
    rois0 = ds.sweep(min_reads=5)
    arrays = util.redraw_mapq(rois0.arrays())
    rois = host.Rois(arrays=arrays)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, arrays, tag="mapq")
    assert cnt["variants"] > 0
    assert_same(dump, vcf, odump, ovcf)
    spread = list(np.linspace(0, 255, 16).astype(int))
    a2 = util.length_fixture([[150] * 16, [150] * 16], seed=5, mapqs=[[255], spread])
    dump, vcf, odump, ovcf, _, _ = run_both(host.Rois(arrays=a2), a2, tag="mapq_directed", **DIRECTED)
    assert_same(dump, vcf, odump, ovcf)


# ---- 3. status bits -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cap", [192, 256, 4096])
def test_contig_overflow_exactly_at_the_cap(cap, capfd):
    """contigs of exactly cap bases are called, cap + 1 bases drop the region: through a merge and, where a read can be that long, through the
    trimmed read itself"""
    arrays = util.cap_fixture(cap)
    lim = util.limits(orc.call(arrays, dump_level=util.DUMP_LIMITS, **DIRECTED)[0])
    flagged = {k for k, (ln, _) in lim.items() if ln > cap}
    assert len(flagged) == (2 if cap < 512 else 1)
    vcf, dump, counts = _device(arrays, max_contig_len=cap, **DIRECTED)
    assert_flagged_exactly(arrays, flagged, RS_CONTIG_OVERFLOW, capfd, dump, vcf, counts, **DIRECTED)


def test_corr_overflow_at_129_voting_sites(capfd):
    """two contigs of four reads merge in the first combine pass with exactly 128 voting sites (called) and 129 (the region is dropped with
    IDL_RS_CORR_OVERFLOW: the device keeps IDL_MAX_CORRECTIONS = 128 sites per merge)"""
    arrays = util.corr_fixture((128, 129, 127))
    lim = util.limits(orc.call(arrays, dump_level=util.DUMP_LIMITS, **DIRECTED)[0])
    assert [lim[k][1] for k in range(3)] == [128, 129, 127]
    vcf, dump, counts = _device(arrays, **DIRECTED)
    assert_flagged_exactly(arrays, {1}, RS_CORR_OVERFLOW, capfd, dump, vcf, counts, **DIRECTED)


def test_dp_overflow_at_call_site_a(capfd):
    """max_contig_len = 8192.  A contig of ~5.9 kb against a ~6 kb window needs exact scores beyond kernel 2's uint16 window: the alignment
    carries IDL_RS_DP_OVERFLOW (region bit 4, counted and named; not a dropping status), it returns no CIGAR, so it has no events and no VCF
    record.  The region's contigs and the other region -- a ~4.9 kb contig just under the window, the longest alignment the path runs,
    whose reversed copy spills from the 448-base shared stage to global memory -- equal the oracle's records"""
    arrays = util.long_contig_fixture((6000, 4900))
    vcf, dump, counts = _device(arrays, max_contig_len=8192, **DIRECTED)
    odump, ovcf, cnt = orc.call(arrays, dump_level=31, use_ref_ksw2=orc.have_ref(), **DIRECTED)
    assert cnt["dp_a"] == 2
    g, o = util.by_region(dump), util.by_region(odump)
    assert g[1] == o[1]
    assert [l for l in g[0] if l[0] in "RC"] == [l for l in o[0] if l[0] in "RC"]
    ga, oa = [l.split("\t") for l in g[0] if l[0] == "A"], [l.split("\t") for l in o[0] if l[0] == "A"]
    assert len(ga) == len(oa) == 1 and ga[0][:5] == oa[0][:5] and ga[0][-2:] == ["", ""]   # same contig and window, no CIGAR
    assert not any(l[0] == "E" for l in g[0]) and any(l[0] == "E" for l in o[0])
    assert counts[RS_DP_OVERFLOW] == 1 and sum(counts) == 1
    assert "DP workspace" in capfd.readouterr().err
    _, ovcf1, _ = orc.call(util.region_subset(arrays, [1]), dump_level=0, use_ref_ksw2=orc.have_ref(), **DIRECTED)
    assert vcf == ovcf1


def test_contig_overflow_on_generator_regions(capfd):
    """150-base reads: every region of this slice grows a contig past 192 bases, so the caps are 256 (57 of 66 regions dropped) and 320 (3
    dropped), on either side of the regions' longest contigs"""
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=60, max_indel=40, tr_fraction=0.3, seed=91)
    rois = ds.sweep(min_reads=5)
    arrays = rois.arrays()
    kw = dict(min_reads=5, min_ctg_len=73, min_event_len=5)
    lim = util.limits(orc.call(arrays, dump_level=util.DUMP_LIMITS, **kw)[0])
    for cap in (256, 320):
        flagged = {k for k, (ln, _) in lim.items() if ln > cap}
        assert 3 <= len(flagged) <= len(lim) - 3
        vcf, dump, counts = _device(arrays, max_contig_len=cap, **kw)
        assert_flagged_exactly(arrays, flagged, RS_CONTIG_OVERFLOW, capfd, dump, vcf, counts, **kw)


def test_region_deeper_than_the_context_refuses_the_batch():
    """n_reads + 2 > max_reads_per_region + 2 slots: idl_submit returns IDL_E_CAPACITY, and the same context then calls the next batch"""
    arrays = util.length_fixture([[150] * 30, [150] * 10])
    shallow = util.region_subset(arrays, [1])
    caller = api.Caller(0, out_flags=abi.OUT_SUPPORT, max_reads_per_region=20, **DIRECTED)
    try:
        with pytest.raises(cuda.IdlError, match="capacity"):
            caller.call(host.Rois(arrays=arrays))
        vcf, dump = caller.call(host.Rois(arrays=shallow), dump_level=31)
    finally:
        caller.close()
    odump, ovcf, _ = orc.call(shallow, dump_level=31, use_ref_ksw2=orc.have_ref(), **DIRECTED)
    assert dump == odump and vcf == ovcf and "\nC\t" in "\n" + dump


def _round64(x):
    return (int(x) + 63) & ~63


@pytest.mark.parametrize("case", ["misaligned", "trim_past_end", "longer_than_max_read_len", "span_past_pool"])
def test_bad_input_drops_only_its_region(case, capfd):
    """a hand-edited read record of region 1 (the bytes it points to stay inside the pools, so a missed check gives a wrong result, not a
    fault): region 1 is dropped with IDL_RS_BAD_INPUT and the other regions give the records of the unedited batch"""
    arrays = util.length_fixture([[150] * 8, [150] * 8, [150] * 8])
    rois = host.Rois(arrays=arrays)
    params = abi.default_params(out_flags=abi.OUT_SUPPORT, **DIRECTED)
    ctx = cuda.Context(0, params)
    n = rois.n_rois
    nr, sb, rb = rois.pack_size(0, n, params)
    b = ctx.batch_alloc(n + 8, nr + 8, sb + 64, rb + 64)
    try:
        rois.pack(0, n, params, b)
        writer = host.VcfWriter()
        t = ctx.submit(b); v0, d0 = writer.records(rois, 0, params, ctx.wait(t), 31); ctx.release(t)
        c = b.contents
        rd = np.ctypeslib.as_array(c.read, shape=(c.n_reads,))
        rg = np.ctypeslib.as_array(c.region, shape=(c.n_regions,))
        j = int(rg["read_begin"][1]) + 3
        if case == "misaligned":
            rd["seq_off"][j] += 1
        elif case == "trim_past_end":
            rd["trim_len"][j] = rd["len"][j] - rd["trim_a"][j] + 1
        elif case == "longer_than_max_read_len":
            rd["len"][j] = params.max_read_len + 1
        else:
            rd["seq_off"][j] = c.n_seq_bases - _round64(rd["len"][j]) + 64
        writer = host.VcfWriter()
        t = ctx.submit(b); v1, d1 = writer.records(rois, 0, params, ctx.wait(t), 31); ctx.release(t)
        counts = list(writer.status_counts())
    finally:
        ctx.batch_free(b); ctx.close()
    odump, ovcf, _ = orc.call(arrays, dump_level=31, use_ref_ksw2=orc.have_ref(), **DIRECTED)
    assert d0 == odump and v0 == ovcf
    assert_flagged_exactly(arrays, {1}, RS_BAD_INPUT, capfd, d1, v1, counts, **DIRECTED)


# ---- 4. deep regions and the workspace budget -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_reads_per_region", [1200, 4000])
def test_regions_of_601_to_1200_reads(max_reads_per_region):
    ds = util.small_dataset("panel500_lowerr", chrom_len=60_000, n_events=6, coverage=600.0, seed=5)
    rois = ds.sweep(min_reads=5, max_read_coverage=1200)
    a = rois.arrays()
    assert (a["roi_n_reads"] > 600).sum() >= 2 and a["roi_n_reads"].max() <= 1200
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, a, tag="deep%d" % max_reads_per_region, max_reads_per_region=max_reads_per_region)
    assert_same(dump, vcf, odump, ovcf)


def test_panel_in_one_batch_at_the_largest_capacities():
    """panel500_lowerr (413 regions of more than 126 reads) in one batch at max_reads_per_region = 4000 and at max_contig_len = 32768: the
    assembler launches as many CTAs as its 32-bit arena offsets allow instead of refusing the batch"""
    ds = util.small_dataset("panel500_lowerr")
    rois = ds.sweep(min_reads=5)
    _, ovcf, cnt = orc.call(rois.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=0, n_threads=os.cpu_count() or 1,
                            use_ref_ksw2=orc.have_ref())
    assert cnt["variants"] > 200
    for kw in (dict(max_reads_per_region=4000), dict(max_contig_len=32768)):
        caller = api.Caller(0, min_reads=5, min_ctg_len=73, min_event_len=5, **kw)
        try:
            tm = []
            vcf, _ = caller.call(rois, timings=tm)
        finally:
            caller.close()
        assert len(tm) == 1 and vcf == ovcf, kw


@pytest.mark.parametrize("budget_mb,ok", [(64, True), (1, False)])
def test_workspace_budget(monkeypatch, budget_mb, ok):
    """a small kernel-2 workspace budget launches fewer groups and computes the same bytes; one CTA's workspaces over the budget is
    IDL_E_CAPACITY"""
    monkeypatch.setenv("IDL_WS_BUDGET_MB", str(budget_mb))
    ds = util.small_dataset("pr1", chrom_len=150_000, n_events=30, max_indel=40, tr_fraction=0.5, tr_max_unit=4, seed=17)
    rois = ds.sweep(min_reads=5)
    if not ok:
        caller = api.Caller(0, min_reads=5, min_ctg_len=73, min_event_len=5)
        try:
            with pytest.raises(cuda.IdlError, match="capacity"):
                caller.call(rois)
        finally:
            caller.close()
        return
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag="budget")
    assert cnt["dp_b"] > 0 and cnt["dp_a"] > 0
    assert_same(dump, vcf, odump, ovcf)
