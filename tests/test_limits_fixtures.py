"""The fixtures of test_gpu_limits.py on the CPU: the oracle's limit lines (dump bit 64, which the device never sets) show that each directed
region sits exactly where it was built to sit, the limit lines change nothing else in the dump, and the redrawn MAPQs reach the k-mer medians
at many distinct values."""
import numpy as np
import pytest

import idl_testutil as util
from oracle import pyoracle as orc

LEN_SETS = [[160, 161] * 4, [27, 28, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257] + [150] * 4]


def test_limit_lines_change_nothing_else():
    a = util.cap_fixture(192)
    d0, v0, _ = orc.call(a, min_reads=3, min_event_len=4, dump_level=31)
    d1, v1, _ = orc.call(a, min_reads=3, min_event_len=4, dump_level=31 | util.DUMP_LIMITS)
    assert v0 == v1 and not any(l.startswith("L\t") for l in d0.splitlines())
    assert "".join(l + "\n" for l in d1.splitlines() if not l.startswith("L\t")) == d0


@pytest.mark.parametrize("cap", [192, 256, 4096])
def test_cap_fixture_sits_on_the_cap(cap):
    a = util.cap_fixture(cap)
    d, v, cnt = orc.call(a, min_reads=3, min_event_len=4, dump_level=31 | util.DUMP_LIMITS)
    lim = util.limits(d)
    want = [cap, cap + 1] + ([cap, cap + 1] if cap < 512 else [])
    assert [lim[k][0] for k in range(len(want))] == want
    assert lim[len(want)][0] <= 192 and v.count("\n") == 1   # the deletion region fits every cap and is called
    assert cnt["vote_invariant_violations"] == 0


def test_length_fixture_reaches_the_kernel_boundaries():
    a = util.length_fixture(LEN_SETS)
    lens = a["len"]
    for n in (27, 28, 63, 64, 65, 127, 128, 129, 160, 161, 192, 193):
        assert n in lens
    d, v, cnt = orc.call(a, min_reads=3, min_event_len=4, dump_level=31)
    assert cnt["al_events"] >= 2 and cnt["dp_b"] > 0 and v.count("\n") == 2


def test_redrawn_mapq_reaches_many_medians():
    ds = util.small_dataset("pr1", chrom_len=300_000, n_events=60, max_indel=40, tr_fraction=0.3, seed=81)
    rois = ds.sweep(min_reads=5)   # owns the memory the arrays view
    a = util.redraw_mapq(rois.arrays())
    assert set(np.unique(a["mapq"])) >= {5, 6, 9, 10, 19, 20, 255}
    d, _, _ = orc.call(a, min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=8)
    E = [l.split("\t") for l in d.splitlines() if l.startswith("E\t")]
    med = {int(f[26]) for f in E} | {int(f[27]) for f in E}
    assert len(med - {-1}) >= 20 and max(med) > 60
    assert any(int(f[22]) > 0 and int(f[22]) % 2 == 0 for f in E)   # an even count of counted reads: the median is the lower middle


def test_mapq_fixture_medians():
    """the directed MAPQ regions: every read at 255, and MAPQs spread evenly over 0-255"""
    spread = list(np.linspace(0, 255, 16).astype(int))
    a = util.length_fixture([[150] * 16, [150] * 16], seed=5, mapqs=[[255], spread])
    d, v, _ = orc.call(a, min_reads=3, min_event_len=4, dump_level=8)
    E = [l.split("\t") for l in d.splitlines() if l.startswith("E\t")]
    assert any(int(f[1]) == 0 and int(f[26]) == 255 for f in E)
    assert any(int(f[1]) == 1 and 0 < int(f[26]) < 255 for f in E)


def test_corr_fixture_sits_on_the_bound():
    a = util.corr_fixture((128, 129, 127))
    d, v, cnt = orc.call(a, min_reads=3, min_event_len=4, dump_level=31 | util.DUMP_LIMITS)
    assert [util.limits(d)[k][1] for k in range(3)] == [128, 129, 127]
    assert cnt["corrections"] == 128 + 129 + 127 and cnt["vote_invariant_violations"] == 0


def test_long_contig_fixture_straddles_the_score_window():
    """call-site A keeps exact scores below 0xF000: (qlen + tlen + 2)(q + e) + min(qlen, tlen) * match, q + e = 5 (ksw2.cuh)"""
    a = util.long_contig_fixture((6000, 4900))
    d, _, cnt = orc.call(a, min_reads=3, min_event_len=4, dump_level=31)
    A = {int(l.split("\t")[1]): l.split("\t") for l in d.splitlines() if l.startswith("A\t")}
    C = {int(l.split("\t")[1]): int(l.split("\t")[5]) for l in d.splitlines() if l.startswith("C\t")}
    need = {k: (C[k] + int(A[k][4]) + 2) * 5 + min(C[k], int(A[k][4])) for k in A}
    assert need[0] >= 0xF000 > need[1] and C[1] > 448
    assert sum(l.startswith("E\t0\t") for l in d.splitlines()) >= 1


def test_read_length_limit_is_refused_by_idl_create():
    """the unbanded call-site B stages trimmed reads of up to 960 bases in shared memory; idl_create refuses a larger max_read_len before
    it looks for a device, so this needs no GPU"""
    from indelope_b200 import abi, cuda
    for n, ok in ((960, True), (961, False), (4096, False)):
        with pytest.raises(cuda.IdlError) as e:
            cuda.Context(0, abi.default_params(max_read_len=n))
            raise cuda.IdlError("created")   # a device was found: the parameters were accepted
        assert ("bad argument" in str(e.value)) != ok
    with pytest.raises(cuda.IdlError) as e:   # banded call-site B stages a band, not the read: 4096 bases are accepted
        cuda.Context(0, abi.default_params(max_read_len=4096, b_bw=50))
        raise cuda.IdlError("created")
    assert "bad argument" not in str(e.value)
