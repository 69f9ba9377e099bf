"""The calling path at chromosome ends, window edges and pool padding against the oracle: the directed edge fixtures (idl_testutil.edge_fixtures,
whose paths test_edge_fixtures.py checks on the CPU) bit for bit in one batch and split over many, the same fixtures as FASTA + BAM through the
device decoder, sweep and batch builder, other command-line values, batches whose padding holds random bases instead of zeros, the resident
leg the benchmark times, and kernel 2 with empty sides."""
import os

import numpy as np
import pytest

import idl_testutil as util
from indelope_b200 import abi, api, cuda, host
from oracle import pyoracle as orc
from test_edge_fixtures import EDGE_PARAMS, K, parse_dump
from test_gpu_bam import _compare_device_and_host_pack
from test_gpu_pipeline import assert_same, run_both

pytestmark = pytest.mark.gpu

COUNTERS = ("n_contigs n_alns n_events n_cigar_ops n_contig_bases offsets_tested dp_cells_a dp_cells_b dp_a dp_b kmer_reads kmer_bytes al_events "
            "kernel_launches").split()


@pytest.mark.parametrize("max_reads", [400_000, 20])
def test_edge_fixtures_bit_exact(max_reads):
    """one batch, and batches of at most 20 reads: every chromosome, and the end of chrA with the start of chrB, split across batches"""
    fx = util.edge_fixtures()
    rois, arrays = util.edge_rois(fx)
    plans = api.plan_batches(rois, 0, rois.n_rois, max_reads=max_reads)
    first_b = fx["regions"].index((1, 0, 45))
    assert len(plans) == 1 if max_reads > 1000 else (len(plans) >= 6 and first_b in [a for a, _ in plans])
    dump, vcf, odump, ovcf, cnt, tm = run_both(rois, arrays, tag="edges_%d" % max_reads, max_reads=max_reads, **EDGE_PARAMS)
    assert len(tm) == len(plans)
    assert cnt["al_events"] > 0 and cnt["variants"] > 0
    assert_same(dump, vcf, odump, ovcf)


def test_edge_files_through_the_device_decoder(tmp_path):
    """the fixtures as FASTA + BAM (S operations before position 0 and past the end): idl_bam_sweep == the host sweep on every target, regions
    touching position 0 and the last base, idl_bam_pack == idlh_pack byte for byte, and the VCF of idl_bam_submit == the oracle's"""
    fx = util.edge_fixtures()
    fa, bam = util.edge_files(fx, tmp_path)
    full = host.Dataset.load(fa, bam)
    rois = full.sweep(min_reads=3)
    a = rois.arrays()
    b = cuda.Bam(open(bam, "rb").read())
    touch0 = touch_end = 0
    for c in range(b.n_ref):
        s = b.sweep(c, min_event_support=3, min_read_coverage=3)
        sel = a["roi_chrom"] == c
        assert np.array_equal(s["roi_start"], a["roi_start"][sel]) and np.array_equal(s["roi_end"], a["roi_stop"][sel])
        begin = int(a["roi_read_begin"][sel][0]) if sel.any() else 0
        assert np.array_equal(s["read_idx"], a["read_idx"][begin:begin + len(s["read_idx"])])
        touch0 += int(np.sum(s["roi_start"] == 0)); touch_end += int(np.sum(s["roi_end"] >= b.ref_len[c] - 1))
    b.close()
    assert touch0 >= 2 and touch_end >= 2
    rois2, vcf = _compare_device_and_host_pack(fa, bam, min_reads=3)
    _, ovcf, cnt = orc.call(rois2.arrays(), dump_level=0, use_ref_ksw2=orc.have_ref(), **EDGE_PARAMS)
    assert vcf == ovcf and cnt["variants"] > 0


@pytest.mark.parametrize("min_reads,min_ctg_len,min_event_len", [(1, 20, 1), (2, 26, 2), (3, 27, 3), (8, 150, 10)])
def test_other_command_line_values(min_reads, min_ctg_len, min_event_len):
    """-m/-c/-e other than the two sets the other tests run: -c below K sends contigs shorter than a k-mer to kernel 2 (contig-side reject 11)"""
    ds = util.small_dataset("pr1", chrom_len=250_000, n_events=50, max_indel=40, tr_fraction=0.3, n_base_rate=0.0005, seed=61)
    rois = ds.sweep(min_reads=min_reads)
    kw = dict(min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len)
    dump, vcf, odump, ovcf, cnt, _ = run_both(rois, rois.arrays(), tag="cli_%d_%d_%d" % (min_reads, min_ctg_len, min_event_len), **kw)
    assert cnt["regions"] > 20 and cnt["variants"] > 0
    assert_same(dump, vcf, odump, ovcf)
    erois, earrays = util.edge_rois(util.edge_fixtures())
    dump, vcf, odump, ovcf, cnt, _ = run_both(erois, earrays, tag="cli_edges_%d_%d_%d" % (min_reads, min_ctg_len, min_event_len), **kw)
    assert_same(dump, vcf, odump, ovcf)
    if min_ctg_len < K:
        clen, _, E = parse_dump(odump)
        assert any(e["reject"] == 11 and e["qstart"] < 0 and clen[(e["region"], e["ci"])] < K for e in E)


# ---- one batch: the edge fixtures + a generator slice with N bases ---------------------------------------------------------------------------------
def _edge_and_n_rois():
    ds = util.small_dataset("pr1", chrom_len=80_000, n_events=16, max_indel=40, n_base_rate=0.002, seed=71)
    g = ds.sweep(min_reads=3)
    ga = g.arrays()
    seq = ga["chrom_seqs"][0].copy()
    rois, arrays = util.edge_rois(util.edge_fixtures(), extra=("chrN", seq, {k: v.copy() if hasattr(v, "copy") else v for k, v in ga.items()}))
    assert b"N" in bytes(arrays["bases"])
    return rois, arrays


def _run(ctx, rois, params, batch, submit=True):
    t = ctx.submit(batch) if submit else ctx.run_resident(batch)
    r = ctx.wait(t)
    c = r.contents
    counters = {k: getattr(c, k) for k in COUNTERS}
    out = host.VcfWriter().records(rois, 0, params, r, 31) if submit else None
    ctx.release(t)
    return out, counters


def _round64(x):
    return (np.asarray(x, np.int64) + 63) & ~63


def _poison_pool(p2, pn, ranges, n_bases, rng):
    """random 2-bit codes at the base positions of `ranges` (list of (begin, end)) and in the 16 slack bytes behind each pool; N bits only where
    the code is 0 (the batch contract of include/indelope_cuda.h)"""
    pos = np.concatenate([np.arange(a, b, dtype=np.int64) for a, b in ranges if b > a] + [np.arange(n_bases, n_bases + 64, dtype=np.int64)])
    code = rng.integers(0, 4, len(pos)).astype(np.uint32)
    nbit = (rng.random(len(pos)) < 0.5) & (code == 0)
    w, sh = pos >> 4, (2 * (pos & 15)).astype(np.uint32)
    np.bitwise_and.at(p2, w, ~(np.uint32(3) << sh))
    np.bitwise_or.at(p2, w, code << sh)
    nw, nsh = pos >> 5, (pos & 31).astype(np.uint32)
    np.bitwise_and.at(pn, nw, ~(np.uint32(1) << nsh))
    np.bitwise_or.at(pn, nw, nbit.astype(np.uint32) << nsh)
    tail = np.arange(n_bases + 64, n_bases + 128, dtype=np.int64)           # the rest of the N plane's slack bytes
    np.bitwise_or.at(pn, tail >> 5, (rng.random(len(tail)) < 0.5).astype(np.uint32) << (tail & 31).astype(np.uint32))
    return len(pos)


def poison(batch, seed=5):
    """overwrite every base position a batch does not use with random bases: [len, round64(len)) of every read, [ref_len, round64(ref_len)) of
    every window, the slack words behind the pools"""
    c = batch.contents
    rng = np.random.default_rng(seed)
    rd = np.ctypeslib.as_array(c.read, shape=(c.n_reads,))
    rg = np.ctypeslib.as_array(c.region, shape=(c.n_regions,))
    seq2 = np.ctypeslib.as_array(c.seq2, shape=(c.n_seq_bases // 16 + 4,)); seqn = np.ctypeslib.as_array(c.seqn, shape=(c.n_seq_bases // 32 + 4,))
    ref2 = np.ctypeslib.as_array(c.ref2, shape=(c.n_ref_bases // 16 + 4,)); refn = np.ctypeslib.as_array(c.refn, shape=(c.n_ref_bases // 32 + 4,))
    so, ln = rd["seq_off"].astype(np.int64), rd["len"].astype(np.int64)
    ro, rl = rg["ref_off"].astype(np.int64), rg["ref_len"].astype(np.int64)
    n1 = _poison_pool(seq2, seqn, list(zip(so + ln, so + _round64(ln))), c.n_seq_bases, rng)
    n2 = _poison_pool(ref2, refn, list(zip(ro + rl, ro + _round64(rl))), c.n_ref_bases, rng)
    return n1, n2


@pytest.mark.parametrize("out_flags", [abi.OUT_SUPPORT, 0])
def test_poisoned_padding_changes_nothing(out_flags):
    """the bases between a record's end and the next 64-base boundary are zero (A) in both packers; kernels that load whole words past a record's
    end (the k-mer pass, the assembler's block screen, the DP staging) must not depend on them: with random bases there, every record, the VCF
    and every work counter stay the same"""
    rois, arrays = _edge_and_n_rois()
    params = abi.default_params(out_flags=out_flags, **EDGE_PARAMS)
    ctx = cuda.Context(0, params)
    n = rois.n_rois
    nr, sb, rb = rois.pack_size(0, n, params)
    b = ctx.batch_alloc(n + 8, nr + 8, sb + 64, rb + 64)
    try:
        rois.pack(0, n, params, b)
        (v0, d0), c0 = _run(ctx, rois, params, b)
        odump, ovcf, _ = orc.call(arrays, dump_level=31, use_ref_ksw2=orc.have_ref(), **EDGE_PARAMS)
        assert v0 == ovcf and "N" in d0
        if out_flags:
            assert d0 == odump
        n1, n2 = poison(b)
        assert n1 > 1000 and n2 > 100
        (v1, d1), c1 = _run(ctx, rois, params, b)
        if d1 != d0:
            with open(os.path.join(util.out_dir(), "diff_poison_%d.txt" % out_flags), "w") as f:
                f.write(util.diff_lines(d0, d1, limit=40))
        assert c1 == c0
        assert d1 == d0 and v1 == v0
    finally:
        ctx.batch_free(b); ctx.close()


def test_resident_leg_counts_what_submit_counts():
    """idl_upload + idl_run_resident (the leg behind bench.py's value): the same work counters as idl_submit on the same batch, twice; a
    submit afterwards (lane 0 is shared) still returns the same records"""
    rois, arrays = _edge_and_n_rois()
    params = abi.default_params(out_flags=abi.OUT_SUPPORT, **EDGE_PARAMS)
    ctx = cuda.Context(0, params)
    n = rois.n_rois
    nr, sb, rb = rois.pack_size(0, n, params)
    b = ctx.batch_alloc(n + 8, nr + 8, sb + 64, rb + 64)
    try:
        rois.pack(0, n, params, b)
        (v0, d0), c0 = _run(ctx, rois, params, b)
        assert c0["al_events"] > 0 and c0["dp_b"] > 0
        ctx.upload(b)
        for _ in range(2):
            _, c = _run(ctx, rois, params, b, submit=False)
            assert c == c0
        (v1, d1), c1 = _run(ctx, rois, params, b)
        assert (v1, d1) == (v0, d0) and c1 == c0
    finally:
        ctx.batch_free(b); ctx.close()


@pytest.mark.parametrize("gapo,w,zdrop", [(4, 50, 400), (5, -1, -1)])
def test_kernel2_empty_sides(gapo, w, zdrop):
    """pairs with an empty query, an empty target or both, mixed with ordinary pairs (the pipeline hands kernel 2 an empty target when a contig
    starts before its region's window): zero-length offsets in idl_ksw2_batch, the early exit (status 1) of the oracle, and the pairs around them
    unchanged"""
    rng = np.random.default_rng(97 + gapo)
    qs, ts = [], []
    for k in range(60):
        base = rng.integers(0, 4, 400).astype(np.uint8)
        q, t = base[:int(rng.integers(1, 200))].copy(), base[:int(rng.integers(1, 300))].copy()
        shape = k % 4
        if shape == 1:
            q = q[:0]
        elif shape == 2:
            t = t[:0]
        elif shape == 3 and k % 8 == 3:
            q, t = q[:0], t[:0]
        qs.append(q); ts.append(t)
    ctx = cuda.Context(0)
    try:
        f, c, extra, _ = ctx.ksw2_batch(qs, ts, gapo=gapo, gape=1, w=w, zdrop=zdrop)
        impls = ["lane", "ref"] if orc.have_ref() else ["lane"]
        for i, (q, t) in enumerate(zip(qs, ts)):
            for impl in impls:
                fo, co, ez = orc.ksw2(q, t, gapo=gapo, gape=1, w=w, zdrop=zdrop, impl=impl)
                assert fo == f[i] and co == c[i], (i, len(q), len(t), impl, fo, f[i])
            if len(q) == 0 or len(t) == 0:
                assert extra[i]["status"] == 1 and extra[i]["cells"] == 0 and f[i]["n_cigar"] == 0
            else:
                assert extra[i]["status"] >= 0
    finally:
        ctx.close()
