"""The whole per-region path on the GPU (through the C ABI: idl_batch_alloc / idl_submit / idl_wait) against the CPU
oracle on the same seeded inputs: contigs (order, start, nreads, sequence, per-base support), ksw_extz_t fields and
CIGARs, event records and counts, and the VCF bytes.  Everything is integer: the bar is bit-exact."""
import os

import numpy as np
import pytest

import idl_testutil as util
from indelope_b200 import abi, host
from oracle import pyoracle as orc

pytestmark = pytest.mark.gpu


def run_both(rois, arrays, min_reads=5, min_ctg_len=73, min_event_len=5, level=31, tag="x", max_reads=400_000, **kw):
    from indelope_b200 import api
    caller = api.Caller(0, min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len, out_flags=abi.OUT_SUPPORT, **kw)
    try:
        tm = []
        vcf, dump = caller.call(rois, dump_level=level, timings=tm, max_reads=max_reads)
    finally:
        caller.close()
    # the oracle runs the reference's own compiled ksw2_extz2_sse.c when oracle/_ref was built (it travels to the GPU box)
    odump, ovcf, cnt = orc.call(arrays, min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len, dump_level=level, use_ref_ksw2=orc.have_ref())
    assert cnt["vote_invariant_violations"] == 0  # the assembler's vote shortcut (assemble.cuh) relies on it
    if dump != odump or vcf != ovcf:
        with open(os.path.join(util.out_dir(), "diff_%s.txt" % tag), "w") as f:
            f.write(util.diff_lines(odump, dump, limit=40) + "\n\nVCF:\n" + util.diff_lines(ovcf, vcf))
        with open(os.path.join(util.out_dir(), "dump_%s_oracle.txt" % tag), "w") as f:
            f.write(odump)
        with open(os.path.join(util.out_dir(), "dump_%s_gpu.txt" % tag), "w") as f:
            f.write(dump)
    return dump, vcf, odump, ovcf, cnt, tm


def lane_counts(arrays, min_reads=5, min_ctg_len=73, min_event_len=5):
    """work counters of the oracle with its own lane model of the DP (the compiled reference reports no cell counts)"""
    return orc.call(arrays, min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len, dump_level=0, n_threads=os.cpu_count() or 1)[2]


def assert_same(dump, vcf, odump, ovcf):
    g, o = util.by_type(dump), util.by_type(odump)
    for t in "RCAEV":
        assert g.get(t, []) == o.get(t, []), "first diff in %s lines:\n%s" % (t, util.diff_lines("\n".join(o.get(t, [])), "\n".join(g.get(t, [])), 4))
    assert dump == odump
    assert vcf == ovcf


def test_pr1_config_bit_exact():
    """BASELINE config 1: 1 Mb, 30x, 200 planted 5-300 bp indels, --min-event-len 5 --min-reads 5"""
    ds = util.small_dataset("pr1")
    rois = ds.sweep(min_reads=5)
    dump, vcf, odump, ovcf, cnt, tm = run_both(rois, rois.arrays(), tag="pr1")
    assert cnt["variants"] >= 15 and cnt["dp_b"] > 0  # the AL fallback is exercised
    assert_same(dump, vcf, odump, ovcf)
    # device work counters agree with the oracle's algorithmic counts (SURVEY 8d)
    assert sum(t["offsets_tested"] for t in tm) == cnt["offsets"]
    lc = lane_counts(rois.arrays())
    assert lc["cells_a"] > 0 and lc["cells_b"] > 0
    assert sum(t["dp_cells_a"] for t in tm) == lc["cells_a"] and sum(t["dp_cells_b"] for t in tm) == lc["cells_b"]
    assert sum(t["kmer_bytes"] for t in tm) == cnt["kmer_bytes"]


@pytest.mark.parametrize("name", ["pr1_small", "tandem_small"])
def test_golden_fixtures(name):
    """the committed golden VCFs and record dumps (tools/make_golden.py: the oracle running the reference's own compiled DP) are
    reproduced byte for byte; tandem_small sends 24 events through the AL fallback (1428 unbanded alignments)"""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools"))
    from make_golden import FIXTURES
    gold = os.path.join(os.path.dirname(__file__), "golden", name)
    ds = util.small_dataset("pr1", **FIXTURES[name])
    rois = ds.sweep(min_reads=5)
    from indelope_b200 import api
    caller = api.Caller(0, min_reads=5, min_ctg_len=73, min_event_len=5)
    try:
        vcf, dump = caller.call(rois, dump_level=31)
    finally:
        caller.close()
    assert rois.header() + vcf == open(gold + ".vcf").read()
    assert "\n".join(l for l in dump.splitlines() if l[:1] in "RAEV") + "\n" == open(gold + ".dump").read()


@pytest.mark.parametrize("name,over", [
    ("short_indels", dict(chrom_len=400_000, n_events=80, max_indel=40, seed=5)),
    ("tandem", dict(chrom_len=400_000, n_events=80, max_indel=40, tr_fraction=0.7, tr_max_unit=4, seed=6)),
    ("noisy", dict(chrom_len=300_000, n_events=60, max_indel=50, sub_rate=0.004, seed=7)),
    ("with_n", dict(chrom_len=300_000, n_events=60, max_indel=40, n_base_rate=0.002, seed=8)),
    ("cov100", dict(chrom_len=200_000, n_events=30, max_indel=40, coverage=100.0, tr_fraction=0.3, seed=9)),
])
def test_variants_of_the_generator(name, over):
    ds = util.small_dataset("pr1", **over)
    rois = ds.sweep(min_reads=5)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag=name)
    assert cnt["regions"] > 20
    assert_same(dump, vcf, odump, ovcf)


def test_default_cli_parameters():
    """docopt defaults: -m 3 -c 73 -e 4 (src/indelope.nim:568-570)"""
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=60, max_indel=40, seed=12)
    rois = ds.sweep(min_reads=3)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), min_reads=3, min_ctg_len=73, min_event_len=4, tag="defaults")
    assert_same(dump, vcf, odump, ovcf)


def test_high_coverage_panel_slice():
    """a slice of the 500x panel at the generator's default error rate: hundreds of reads and contigs per region, nearly every region
    dies at the 20-contig gate of src/indelope.nim:209 -- this one checks kernel 1 on deep regions and the gate itself"""
    ds = util.small_dataset("panel500", chrom_len=120_000, n_events=14, coverage=300.0)
    rois = ds.sweep(min_reads=5)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag="panel")
    assert cnt["contigs_pre"] > 20 * cnt["regions"]
    assert_same(dump, vcf, odump, ovcf)


@pytest.mark.parametrize("over,min_dp_b", [
    (dict(chrom_len=120_000, n_events=14, coverage=300.0), 3000),
    (dict(chrom_len=100_000, n_events=10, coverage=420.0, seed=77), 2000),
])
def test_deep_regions_reach_alignment_and_the_al_fallback(over, min_dp_b):
    """deep regions (every one > 126 reads: assemble_kernel<256>) that SURVIVE the 20-contig gate: contig alignment, k-mer counting
    and the AL fallback with hundreds of reads per event (SURVEY.md 8d.4: the survivors of the panel)"""
    ds = util.small_dataset("panel500_lowerr", **over)
    rois = ds.sweep(min_reads=5)
    a = rois.arrays()
    assert a["roi_n_reads"].min() > 126
    dump, vcf, odump, ovcf, cnt, tm = run_both(rois, a, tag="deep_al")
    assert cnt["dp_a"] > 0 and cnt["dp_b"] > min_dp_b and cnt["al_events"] > 0 and cnt["variants"] > 0
    assert sum(t["dp_b"] for t in tm) == cnt["dp_b"] and sum(t["al_events"] for t in tm) == cnt["al_events"]
    assert_same(dump, vcf, odump, ovcf)


def test_many_small_batches_keep_order_and_dedup():
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=60, max_indel=40, seed=13)
    rois = ds.sweep(min_reads=5)
    from indelope_b200 import api
    caller = api.Caller(0, min_reads=5, min_ctg_len=73, min_event_len=5)
    try:
        v1, _ = caller.call(rois)
        v2, _ = caller.call(rois, max_reads=300)  # dozens of batches over both lanes
    finally:
        caller.close()
    _, ovcf, _ = orc.call(rois.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=0, use_ref_ksw2=orc.have_ref())
    assert v1 == ovcf and v2 == ovcf


def test_empty_batch_and_tiny_regions():
    from indelope_b200 import api
    ref = "".join("ACGT"[i] for i in np.random.default_rng(1).integers(0, 4, 3000))
    reads = [dict(start=1000 + i, seq=ref[1000 + i:1150 + i]) for i in range(0, 50, 10)]
    rois, arrays = util.rois_from_reads(reads, ref)
    dump, vcf, odump, ovcf, _, _ = run_both(rois, arrays, min_reads=3, tag="tiny")
    assert_same(dump, vcf, odump, ovcf)
    caller = api.Caller(0)
    try:
        v, d = caller.call(rois, lo=0, hi=0)
        assert v == "" and d == ""
    finally:
        caller.close()


@pytest.mark.parametrize("read_len", [100, 250])
def test_other_read_lengths(read_len):
    """100 bp and 250 bp reads: the unbanded AL alignments then need one / three trips of packed words per diagonal"""
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=50, max_indel=40, read_len=read_len, tr_fraction=0.3, seed=31 + read_len)
    rois = ds.sweep(min_reads=5)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag="len%d" % read_len)
    assert cnt["regions"] > 20 and cnt["dp_b"] > 0
    assert_same(dump, vcf, odump, ovcf)


def test_deep_regions_use_the_cta_assembler():
    """regions with more than 126 reads (up to the 600-read cap of src/indelope.nim:515) go through assemble_kernel<256>"""
    ds = util.small_dataset("panel500", chrom_len=100_000, n_events=10, coverage=420.0, seed=77)
    rois = ds.sweep(min_reads=5)
    a = rois.arrays()
    assert a["roi_n_reads"].max() > 400 and a["roi_n_reads"].max() <= 600
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, a, tag="deep")
    assert cnt["contigs_pre"] > 20 * cnt["regions"]  # kernel 1 only: these regions stop at the 20-contig gate (the AL-heavy deep case is the test above)
    assert_same(dump, vcf, odump, ovcf)


def _random_seq(rng, n):
    return "".join("ACGT"[i] for i in rng.integers(0, 4, n))


def test_directed_gates_and_odd_reads():
    """directed regions for paths random data rarely hits: an empty first read (all qualities below 15), MAPQ at the 20/10/5
    gates, exactly 20 and 21 pre-combine contigs (src/indelope.nim:209), a read shorter than K, a skippable read, Ns"""
    rng = np.random.default_rng(123)
    ref = _random_seq(rng, 6000)
    sets = []
    for n_single in (18, 19):  # 1 empty + 1 merged contig + n singletons = 20 / 21 pre-combine contigs
        reads = []
        base = 2000
        hap = ref[base:base + 70] + ref[base + 82:base + 400]  # 12 bp deletion
        reads.append(dict(start=base, seq=ref[base:base + 150], qual=[2] * 150))                       # trimmed to nothing: empty first contig
        for k in range(4):
            for c in range(5):
                off = 10 * k + c
                reads.append(dict(start=base + off, seq=hap[off:off + 150], mapq=[60, 20, 19, 60, 60][c]))  # 19 is skipped by assemble
        for j in range(n_single):
            reads.append(dict(start=base + 20 + j, seq=_random_seq(rng, 150), mapq=60))                  # singletons
        for j in range(3):
            reads.append(dict(start=base + 40 + j, seq=_random_seq(rng, 150), mapq=9))                   # MAPQ 9: neither assembled nor counted
        reads.append(dict(start=base + 30, seq=ref[base + 30:base + 50]))                              # 20 bp < K: never matches a k-mer
        reads.append(dict(start=base + 31, seq=hap[31:181], flag=0x400))                                # duplicate: skippable
        reads.append(dict(start=base + 32, seq=hap[32:100] + "N" + hap[101:182], mapq=5))               # N base, MAPQ 5 does not extend the window
        reads.sort(key=lambda r: r["start"])
        _, arrays = util.rois_from_reads(reads, ref, roi_start=base + 60, roi_stop=base + 90)
        sets.append(arrays)
    arrays = util.merge_rois(sets)
    rois = host.Rois(arrays=arrays)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, arrays, min_reads=3, min_event_len=4, tag="directed")
    pre = [int(l.split("\t")[2].split("=")[1]) for l in odump.splitlines() if l.startswith("R\t")]
    assert pre == [20, 21], pre   # the two regions straddle the n_contigs > 20 gate
    assert sum(l.startswith("A\t0\t") for l in odump.splitlines()) >= 1 and not any(l.startswith("A\t1\t") for l in odump.splitlines())
    assert_same(dump, vcf, odump, ovcf)


def test_block_screen_edges_short_reads_and_periodic_sequence():
    """the assembler's 32-offset block screen (16 leading bases, position parallel): reads around the min_overlap 16/17
    switch (18-24 bp reads take the per-offset path, longer ones the blocks), and homopolymer / dinucleotide / 7-mer
    repeats where dozens of offsets of one block survive the screen and run the full compare"""
    rng = np.random.default_rng(2024)
    units, rep_lens = ["A", "CA", "GATTACA", "T", "ACG", "AAAC"], [40, 90, 140, 260, 64, 33]
    segs, haps, seg_start, at = [], [], [], 0
    for unit, rl in zip(units, rep_lens):
        left, right = _random_seq(rng, 1500), _random_seq(rng, 1500)
        rep = (unit * 300)[:rl]
        segs.append(left + rep + right)
        haps.append(left + rep[:len(rep) - len(unit) * 3] + right)      # contraction by three units
        seg_start.append(at); at += len(segs[-1])
    ref = "".join(segs)
    sets = []
    for k in range(6):
        base = 1500 - 170
        reads = []
        for i in range(0, 330, 3):
            src = haps[k] if (i // 3) % 2 else segs[k]
            L = [150, 150, 18, 150, 19, 20, 150, 21, 24, 150, 40, 150, 64, 150][(i // 3) % 14]
            reads.append(dict(start=seg_start[k] + base + i, seq=src[base + i:base + i + L], mapq=60))
        reads.sort(key=lambda r: r["start"])
        _, arrays = util.rois_from_reads(reads, ref, roi_start=seg_start[k] + 1500, roi_stop=seg_start[k] + 1500 + rep_lens[k])
        sets.append(arrays)
    arrays = util.merge_rois(sets)
    rois = host.Rois(arrays=arrays)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, arrays, min_reads=3, min_event_len=3, tag="blocks")
    assert cnt["regions"] == 6 and cnt["offsets"] > 10000
    assert_same(dump, vcf, odump, ovcf)


@pytest.mark.parametrize("name", ["exome", "panel500", "panel500_lowerr"])
def test_exome_and_panel_configs_at_full_size(name):
    """BASELINE configs 2 and 4 as host.CONFIGS defines them (100x exome: ~2 900 regions of 100-300 reads; 500x panel: regions at
    the 600-read cap, every one past the 20-contig gate at the default error rate -- kernel 1 only -- and, at 2e-4 substitutions per
    base, 413 deep regions of which most survive: 121 k unbanded alignments from 120 AL events): every record -- contigs with
    per-base support, alignments, events -- and the VCF, bit for bit; the rare assembler paths are seen to fire"""
    ds = util.small_dataset(name)
    rois = ds.sweep(min_reads=5)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag=name)
    assert cnt["regions"] > 400
    if name == "panel500":
        assert cnt["dp_a"] == 0  # as realised, config 4 at the default error rate never reaches kernel 2
    else:
        assert cnt["corrections"] > 0 and cnt["left_merges"] > 0  # voted corrections and left-overhang merges happened
    if name == "panel500_lowerr":
        assert cnt["dp_b"] > 100_000 and cnt["al_events"] > 100 and cnt["variants"] > 200
    assert_same(dump, vcf, odump, ovcf)


@pytest.mark.parametrize("name,min_regions,min_variants", [("chr1", 80_000, 10_000), ("wgs", 40_000, 5_000)])
def test_full_workloads_are_byte_identical_and_batching_invariant(name, min_regions, min_variants):
    """BASELINE config 3 at its full size (the workload bench.py times: 62 000 planted events on a 248 Mb contig, ~85 k regions,
    ~2.5 M reads, ~484 k unbanded and ~128 k banded alignments) and one rank's shard of config 5: the VCF equals the oracle's
    byte for byte, the device work counters equal the oracle's, and cutting the work into finer batches changes nothing"""
    ds = util.small_dataset(name)
    rois = ds.sweep(min_reads=5)
    assert rois.n_rois > min_regions
    from indelope_b200 import api
    caller = api.Caller(0, min_reads=5, min_ctg_len=73, min_event_len=5)
    try:
        tm = []
        v1, _ = caller.call(rois, timings=tm)
        v2, _ = caller.call(rois, max_reads=90_000)
    finally:
        caller.close()
    _, ovcf, cnt = orc.call(rois.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=0, n_threads=os.cpu_count() or 1, use_ref_ksw2=orc.have_ref())
    assert cnt["corrections"] > 0 and cnt["left_merges"] > 0 and cnt["vote_invariant_violations"] == 0
    assert v1 == ovcf
    assert v2 == v1
    assert sum(t["offsets_tested"] for t in tm) == cnt["offsets"]
    lc = lane_counts(rois.arrays())
    assert lc["cells_a"] > 0 and lc["cells_b"] > 0
    assert sum(t["dp_cells_a"] for t in tm) == lc["cells_a"] and sum(t["dp_cells_b"] for t in tm) == lc["cells_b"]
    assert sum(t["dp_b"] for t in tm) == cnt["dp_b"] and sum(t["al_events"] for t in tm) == cnt["al_events"]
    assert cnt["variants"] > min_variants


def test_estimated_pools_grow_instead_of_failing(monkeypatch):
    """the CIGAR pool and the AL item pool are sized from estimates; a batch that needs more is run again inside idl_wait with pools
    sized from the device's own counts (the reference would simply finish): same bytes, and the relaunch is reported"""
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=60, max_indel=40, tr_fraction=0.5, tr_max_unit=4, seed=41)
    rois = ds.sweep(min_reads=5)
    _, ovcf, cnt = orc.call(rois.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=0, use_ref_ksw2=orc.have_ref())
    assert cnt["dp_b"] > 500 and cnt["dp_a"] > 50
    monkeypatch.setenv("IDL_CIGAR_PER_ALN", "0")
    monkeypatch.setenv("IDL_ITEMS_PER_READ", "0")
    from indelope_b200 import api
    caller = api.Caller(0, min_reads=5, min_ctg_len=73, min_event_len=5)
    try:
        tm = []
        vcf, _ = caller.call(rois, timings=tm)
    finally:
        caller.close()
    assert sum(t["pool_retries"] for t in tm) >= 1
    assert vcf == ovcf


def test_status_bits_are_reported_never_silent(capfd):
    """a soft-masked / IUPAC read is folded and the region says so (IDL_RS_ALPHABET, results still produced); a read longer than
    max_read_len drops its region (IDL_RS_READ_TOO_LONG) without failing the batch; the other regions are untouched"""
    rng = np.random.default_rng(99)
    ref = _random_seq(rng, 5000)
    hap = ref[:2070] + ref[2082:]  # 12 bp deletion
    sets = []
    for case in range(3):
        reads = []
        for i in range(0, 120, 4):
            src = hap if (i // 4) % 2 else ref
            reads.append(dict(start=1950 + i, seq=src[1950 + i:2100 + i]))
        if case == 1:
            reads[4]["seq"] = reads[4]["seq"][:30].lower() + reads[4]["seq"][30:]
        if case == 2:
            reads[6] = dict(start=1950 + 24, seq=ref[1974:1974 + 600])
        _, arrays = util.rois_from_reads(reads, ref, roi_start=2060, roi_stop=2090)
        sets.append(arrays)
    arrays = util.merge_rois(sets)
    rois = host.Rois(arrays=arrays)
    from indelope_b200 import api
    caller = api.Caller(0, min_reads=3, min_ctg_len=73, min_event_len=4, out_flags=abi.OUT_SUPPORT)
    try:
        vcf, dump = caller.call(rois, dump_level=31)
        counts = caller.status_counts
    finally:
        caller.close()
    err = capfd.readouterr().err
    assert counts[5] == 1 and counts[4] == 1 and sum(counts) == 2  # bit 5 = IDL_RS_ALPHABET, bit 4 = IDL_RS_READ_TOO_LONG
    assert "folded" in err and "max_read_len" in err
    r = [l for l in dump.splitlines() if l.startswith("R\t")]
    assert len(r) == 3 and r[2].endswith("n=0") and not r[0].endswith("n=0") and not r[1].endswith("n=0")
    # regions 0 and 1 differ only by case: same contigs, same records (the oracle, given the folded text, agrees)
    up = dict(arrays); up["bases"] = np.frombuffer(bytes(arrays["bases"]).upper(), dtype=np.uint8)
    for k in ("roi_chrom", "roi_start", "roi_stop", "roi_read_begin", "roi_n_reads"):
        up[k] = arrays[k][:2]
    odump, ovcf, _ = orc.call(up, min_reads=3, min_ctg_len=73, min_event_len=4, dump_level=31, use_ref_ksw2=orc.have_ref())
    assert "\n".join(l for l in dump.splitlines() if l.split("\t")[1] in ("0", "1") or l.startswith("V")) == odump.rstrip("\n")
    assert vcf == ovcf and vcf.count("\n") == 1  # regions 0 and 1 call the same deletion: the second record falls to the dedup (:604-608)
