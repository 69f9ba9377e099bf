"""kernel 2 (ksw2 extension DP + traceback) through the C ABI (idl_ksw2_batch) against the CPU oracle's lane model
and, when oracle/_ref was built, against the reference's own compiled C file.  Bit-exact: every ksw_extz_t field and
the full CIGAR."""
import numpy as np
import pytest

import idl_testutil as util
from oracle import pyoracle as orc
from test_oracle_ksw2 import QRY, QRY2, TGT, TGT2, random_pair

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from indelope_b200 import cuda
    c = cuda.Context(0)
    yield c
    c.close()


def check(ctx, pairs, impl="lane"):
    """pairs: list of (q codes, t codes); one parameter set per call"""
    (go, w, z) = pairs[0][2:]
    f, c, extra, ms = ctx.ksw2_batch([p[0] for p in pairs], [p[1] for p in pairs], gapo=go, gape=1, w=w, zdrop=z)
    bad = []
    for i, (q, t, _, _, _) in enumerate(pairs):
        fo, co, ez = orc.ksw2(q, t, gapo=go, gape=1, w=w, zdrop=z, impl=impl)
        if extra[i]["status"] < 0:
            bad.append((i, "status", extra[i]["status"], len(q), len(t)))
        elif fo != f[i] or co != c[i] or (impl == "lane" and ez.cells != extra[i]["cells"]):
            bad.append((i, len(q), len(t), fo, f[i], orc.cigar_str(co), orc.cigar_str(c[i])))
    return bad


def test_known_answers(ctx):  # SURVEY appendix F / src/ksw2/ksw2.nim:171-215 with flag 0
    f, c, _, _ = ctx.ksw2_batch([orc.encode(QRY)], [orc.encode(TGT)], gapo=3, gape=1, w=-1, zdrop=-1)
    assert orc.cigar_str(c[0]) == "52M19D41M6D5M22D"
    assert (f[0]["max"], f[0]["max_q"], f[0]["max_t"], f[0]["mqe"], f[0]["mqe_t"], f[0]["mte"], f[0]["mte_q"], f[0]["score"], f[0]["zdropped"]) == (73, 97, 116, 73, 116, 42, 82, 42, 0)
    f, c, _, _ = ctx.ksw2_batch([orc.encode(QRY), orc.encode(QRY2)], [orc.encode(TGT), orc.encode(TGT2)], gapo=4, gape=1, w=50, zdrop=400)
    assert orc.cigar_str(c[0]) == "52M19D46M28D" and (f[0]["max"], f[0]["max_q"], f[0]["max_t"], f[0]["score"]) == (72, 71, 71, 40)
    assert orc.cigar_str(c[1]) == "11D3M1D7M6D16M21D18M1I22M1D17M3D1M" and (f[1]["max"], f[1]["max_q"], f[1]["max_t"], f[1]["score"]) == (0, -1, -1, -75)


def test_edge_shapes(ctx):
    rng = np.random.default_rng(3)
    pairs = []
    for ql, tl in [(1, 1), (1, 40), (40, 1), (15, 16), (16, 15), (17, 33), (150, 150), (31, 500), (200, 17), (64, 64), (65, 129)]:
        base = rng.integers(0, 4, max(ql, tl) + 5).astype(np.uint8)
        pairs.append((base[:ql].copy(), base[:tl].copy(), 4, 50, 400))
    assert check(ctx, pairs) == []
    pairs = [(p[0], p[1], 5, -1, -1) for p in pairs]
    assert check(ctx, pairs) == []


@pytest.mark.parametrize("impl", ["lane", "ref"])
def test_fuzz_bit_exact(ctx, impl):
    if impl == "ref" and not orc.have_ref():
        pytest.skip("oracle/_ref/libksw2_ref.so not built")
    rng = np.random.default_rng(20171101 if impl == "lane" else 77)
    groups = {}
    for _ in range(3000):
        q, t, go, w, z = random_pair(rng)
        groups.setdefault((go, w, z), []).append((q, t, go, w, z))
    bad = []
    for key, pairs in groups.items():
        bad += [(key,) + b for b in check(ctx, pairs, impl)]
    assert bad == [], bad[:5]


def test_production_shapes_many(ctx):
    """call-site A (bw=50, z=400, q=4) and call-site B (unbanded, q=5) shapes of src/indelope.nim:221,343-344"""
    rng = np.random.default_rng(11)
    A, B = [], []
    for _ in range(600):
        ql = int(rng.integers(73, 900)); base = rng.integers(0, 4, ql + 300).astype(np.uint8)
        q = base[:ql].copy(); t = base[:ql + int(rng.integers(64, 250))].copy()
        pos = int(rng.integers(20, ql - 20)); L = int(rng.integers(1, 70))
        q = np.concatenate([q[:pos], rng.integers(0, 4, L).astype(np.uint8), q[pos:]]) if rng.random() < 0.5 else np.concatenate([q[:pos], q[pos + L:]])
        A.append((q, t, 4, 50, 400))
        tl = int(rng.integers(100, 900)); base = rng.integers(0, 4, tl + 200).astype(np.uint8)
        o = int(rng.integers(0, tl - 50)); r = base[o:o + int(rng.integers(30, 151))].copy()
        m = rng.random(len(r)) < 0.01; r[m] = rng.integers(0, 4, int(m.sum()))
        B.append((r, base[:tl].copy(), 5, -1, -1))
    assert check(ctx, A) == []
    assert check(ctx, B) == []


def test_band_leaves_the_matrix_on_the_right(ctx):
    """target much shorter than the query under a band: the last diagonals have a one-column band whose H[en0] is built from
    a column that left the band earlier (the uint16 score ring re-bases it), ksw2_extz2_sse.c:318"""
    rng = np.random.default_rng(5)
    pairs = []
    for ql, tl, w in [(300, 100, 50), (400, 64, 50), (257, 33, 20), (500, 180, 10), (90, 17, 3), (200, 1, 50), (150, 2, 1)]:
        base = rng.integers(0, 4, ql + 10).astype(np.uint8)
        pairs.append((base[:ql].copy(), base[:tl].copy(), 4, w, 10_000))  # z-drop out of the way: run until the band is exhausted
    for p in pairs:  # one parameter set per call
        assert check(ctx, [p]) == []
        assert check(ctx, [(p[0], p[1], 4, p[3], -1)]) == []


def test_long_alignments_and_score_window(ctx):
    """a few kb per side is inside the uint16 score window of the kernel; far beyond it the alignment is reported as a capacity
    status (negative), never returned wrong"""
    rng = np.random.default_rng(9)
    base = rng.integers(0, 4, 4200).astype(np.uint8)
    q = base[:3000].copy(); t = np.concatenate([base[:1500], base[1530:3300]])
    assert check(ctx, [(q, t, 4, 50, 400)]) == []
    assert check(ctx, [(q[:400], t[:1000], 5, -1, -1)]) == []  # unbanded: the whole anti-diagonal lives in the shared-memory rings
    big = rng.integers(0, 4, 9000).astype(np.uint8)
    f, c, extra, _ = ctx.ksw2_batch([big[:4500]], [big[:8200]], gapo=4, gape=1, w=50, zdrop=400)  # (qlen + tlen)(q + e) leaves the window
    assert extra[0]["status"] < 0 and f[0]["n_cigar"] == 0


def test_row_owned_variant_edges(ctx):
    """the unbanded call-site keeps the query rows in registers for reads of up to 256 bases (ksw2_rows.cuh): every row count
    around the word / slot / variant boundaries against short and long targets, tandem repeats and N codes"""
    rng = np.random.default_rng(17)
    pairs = []
    for ql in (1, 2, 3, 4, 5, 7, 8, 31, 32, 33, 127, 128, 129, 150, 159, 160, 161, 200, 255, 256, 257, 300):
        for tl in (1, 2, 3, 4, 5, 17, 149, 233, 700):
            base = rng.integers(0, 4, ql + tl + 8).astype(np.uint8)
            o = int(rng.integers(0, tl))
            q = base[o:o + ql].copy(); t = base[:tl].copy()
            if rng.random() < 0.3:
                unit = rng.integers(0, 4, int(rng.integers(1, 4))).astype(np.uint8)
                k = int(rng.integers(0, max(1, tl - 1))); t[k:k + 20] = np.resize(unit, len(t[k:k + 20]))
            m = rng.random(len(q)) < 0.03; q[m] = rng.integers(0, 5, int(m.sum()))
            pairs.append((q, t, 5, -1, -1))
    for impl in (["lane", "ref"] if orc.have_ref() else ["lane"]):
        assert check(ctx, pairs, impl) == []
    # targets too long for the shared-memory staging of the row-owned variant fall back to the column-owned one, per warp
    long_t = rng.integers(0, 4, 2600).astype(np.uint8)
    mixed = [(long_t[40:190].copy(), long_t[:2500].copy(), 5, -1, -1), (long_t[5:105].copy(), long_t[:1900].copy(), 5, -1, -1)] + pairs[100:110]
    assert check(ctx, mixed) == []
    # other gap costs through the same variant
    assert check(ctx, [(p[0], p[1], 3, -1, -1) for p in pairs[::3]]) == []


def test_row_owned_equals_column_owned(ctx, monkeypatch):
    """IDL_KSW2_COLUMNS=1 keeps unbanded alignments on the column-owned variant: both give the same records and CIGARs"""
    rng = np.random.default_rng(23)
    qs, ts = [], []
    for _ in range(400):
        tl = int(rng.integers(20, 900)); base = rng.integers(0, 4, tl + 260).astype(np.uint8)
        o = int(rng.integers(0, tl)); q = base[o:o + int(rng.integers(1, 257))].copy()
        m = rng.random(len(q)) < 0.02; q[m] = rng.integers(0, 4, int(m.sum()))
        qs.append(q); ts.append(base[:tl].copy())
    a = ctx.ksw2_batch(qs, ts, gapo=5, gape=1, w=-1, zdrop=-1)
    monkeypatch.setenv("IDL_KSW2_COLUMNS", "1")
    b = ctx.ksw2_batch(qs, ts, gapo=5, gape=1, w=-1, zdrop=-1)
    assert a[0] == b[0] and a[1] == b[1]


@pytest.mark.parametrize("match,mismatch,gapo,gape", [(2, -4, 4, 2), (1, -1, 2, 1), (3, -6, 10, 3), (5, -4, 20, 5), (1, -3, 6, 1), (2, -4, 30, 2)])
def test_unbanded_other_scoring_parameters(ctx, match, mismatch, gapo, gape):
    """the unbanded call-site under scoring parameters other than indelope's: the row-owned variant serves every set with
    match + 2(q+e) <= 63 (its carry-free recurrence), the last set exceeds that and falls back to the column-owned variant;
    all against the reference's own compiled C file when it is there, the lane model otherwise"""
    impl = "ref" if orc.have_ref() else "lane"
    rng = np.random.default_rng(1000 + 7 * match + gapo)
    qs, ts = [], []
    for _ in range(160):
        tl = int(rng.integers(1, 500)); base = rng.integers(0, 4, tl + 170).astype(np.uint8)
        o = int(rng.integers(0, tl)); q = base[o:o + int(rng.integers(1, 161))].copy()
        if rng.random() < 0.3:
            unit = rng.integers(0, 4, int(rng.integers(1, 5))).astype(np.uint8); q = np.resize(unit, len(q)).copy()
        m = rng.random(len(q)) < 0.03; q[m] = rng.integers(0, 5, int(m.sum()))
        qs.append(q); ts.append(base[:tl].copy())
    f, c, extra, _ = ctx.ksw2_batch(qs, ts, match=match, mismatch=mismatch, gapo=gapo, gape=gape, w=-1, zdrop=-1)
    bad = []
    for i, (q, t) in enumerate(zip(qs, ts)):
        fo, co, _ = orc.ksw2(q, t, match=match, mismatch=mismatch, gapo=gapo, gape=gape, w=-1, zdrop=-1, impl=impl)
        if extra[i]["status"] < 0 or fo != f[i] or co != c[i]:
            bad.append((i, len(q), len(t), extra[i]["status"], fo, f[i]))
    assert bad == [], bad[:3]


def test_four_threads_per_alignment_equals_eight(ctx, monkeypatch):
    """the banded call-site runs its shared-memory rings with four threads per alignment (eight alignments per warp in lockstep);
    IDL_KSW2_COLUMNS=1 runs it on the eight-thread ring group that call-site B falls back to: same records and CIGARs for ten band
    widths, and the oracle on production parameters"""
    rng = np.random.default_rng(31)
    for w, z in [(50, 400), (100, 400), (7, 100), (33, -1), (200, 50), (79, 400), (80, 400), (1, 100), (17, -1), (33, 60)]:
        qs, ts = [], []
        for _ in range(250):
            ql = int(rng.integers(1, 700)); base = rng.integers(0, 4, ql + 400).astype(np.uint8)
            q = base[:ql].copy(); t = base[:max(1, ql + int(rng.integers(-60, 260)))].copy()
            pos = int(rng.integers(0, max(1, ql - 1))); L = int(rng.integers(1, 90))
            q = np.concatenate([q[:pos], rng.integers(0, 4, L).astype(np.uint8), q[pos:]]) if rng.random() < 0.5 else np.concatenate([q[:pos], q[min(len(q) - 1, pos + L):]])
            m = rng.random(len(q)) < 0.02; q[m] = rng.integers(0, 5, int(m.sum()))
            qs.append(q); ts.append(t)
        a = ctx.ksw2_batch(qs, ts, gapo=4, gape=1, w=w, zdrop=z)
        monkeypatch.setenv("IDL_KSW2_COLUMNS", "1")
        b = ctx.ksw2_batch(qs, ts, gapo=4, gape=1, w=w, zdrop=z)
        monkeypatch.delenv("IDL_KSW2_COLUMNS")
        assert a[0] == b[0] and a[1] == b[1] and a[2] == b[2], (w, z)
    pairs = []
    for _ in range(900):
        q, t, go, w, z = random_pair(rng)
        if w >= 0:
            pairs.append((q, t, 4, 50, 400))
    assert check(ctx, pairs, "ref" if orc.have_ref() else "lane") == []
