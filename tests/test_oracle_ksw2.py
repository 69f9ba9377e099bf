"""ksw2: the oracle's lane model and the reference's own compiled C file.

KATs: src/ksw2/ksw2.nim:166-239 (suite "ksw2 suite") and SURVEY.md appendix F (values obtained by running the
reference C here). Fuzz: lane model == compiled reference on every ksw_extz_t field and the full CIGAR.
"""
import hashlib
import os

import numpy as np
import pytest

from oracle import pyoracle as orc

TGT = "CGAAACTGGGCTACTCCATGACCAGGGGCAAAATAGGCTTTTAGCCGCTGCGTTCTGGGAGCTCCTCCCCCTTCTGGGAGCTCCTCCCCCTCCCCAGAAGGCCAAGGGATGTGGGGGCTGGGGGACTGGGAGGCCTGGCAGTCTT"
QRY = "CGAAACTGGGCTACTCCATGACCAGGGGCAAAATAGGCTTTTAGCCGCTGCGTTCTGGGAGCTCCTCCCCCTCCCCAGAAGGCCAAGGGATGTTGGGG"
TGT2 = "TGGCGCCTTGGCCTACAGGGGCCGCGGTTGAGGGTGGGAGTGGGGGTGCACTGGCCAGCACCTCAGGAGCTGGGGGTGGTGGTGGGGGCGGTGGGGGTGGTGTTAGTACCCCATCTTTTAGGTCTGA"
QRY2 = "CCTCAGGAGCTGGGGGTGGTGGTGGGGGCGGTGGGGGTGGTGTTAGTACCCCATCTTGTAGGTCTGAAACACAAAGTGTGGGGTG"

needs_ref = pytest.mark.skipif(not orc.have_ref(), reason="oracle/_ref/libksw2_ref.so not built")


def trunc(cig, max_q):
    """the `cigar` iterator of src/ksw2/ksw2.nim:22-33"""
    out, off, lim = [], 0, max_q & 0xFFFFFFFF
    for c in cig:
        if off >= lim:
            break
        if (c & 15) != 2:
            off += c >> 4
        out.append(c)
    return out


def test_encode_and_matrix():  # src/ksw2/ksw2.nim:185-192
    assert orc.encode(TGT)[0] == 1 and orc.encode(QRY)[0] == 1 and len(orc.encode(QRY)) == len(QRY)
    assert list(orc.encode("ACGTNacgtnX")) == [0, 1, 2, 3, 4, 0, 1, 2, 3, 4, 4]


@needs_ref
def test_reference_suite_kat():  # src/ksw2/ksw2.nim:176-218: flag = KSW_EZ_EXTZ_ONLY | KSW_EZ_RIGHT, gap_open 3
    f, cig, _ = orc.ksw2(QRY, TGT, gapo=3, gape=1, flag=0x40 | 0x02, impl="ref")
    t = trunc(cig, f["max_q"])
    assert orc.cigar_str(t) == "72M19D26M" and len(t) == 3
    assert f["max_q"] + 1 == 98 and f["max_t"] + 1 == 117 and f["mqe_t"] == 116
    assert max(c >> 4 for c in t if c & 15) == 19
    f, cig, _ = orc.ksw2(QRY2, TGT2, gapo=3, gape=1, flag=0x42, impl="ref")
    assert orc.cigar_str(cig) == "60D67M" and (f["max"], f["max_q"], f["max_t"], f["score"]) == (1, 66, 126, -20)


@pytest.mark.parametrize("impl", ["lane", pytest.param("ref", marks=needs_ref)])
def test_production_parameter_kats(impl):  # SURVEY appendix F
    f, cig, _ = orc.ksw2(QRY, TGT, gapo=3, impl=impl)
    assert orc.cigar_str(cig) == "52M19D41M6D5M22D"
    assert (f["max"], f["max_q"], f["max_t"], f["mqe"], f["mqe_t"], f["mte"], f["mte_q"], f["score"], f["zdropped"]) == (73, 97, 116, 73, 116, 42, 82, 42, 0)
    f, cig, _ = orc.ksw2(QRY, TGT, gapo=4, gape=1, w=50, zdrop=400, impl=impl)
    assert orc.cigar_str(cig) == "52M19D46M28D"
    assert (f["max"], f["max_q"], f["max_t"], f["mqe"], f["mqe_t"], f["mte"], f["score"]) == (72, 71, 71, 72, 116, 40, 40)
    assert orc.cigar_str(trunc(cig, f["max_q"])) == "52M19D46M"
    f, cig, _ = orc.ksw2(QRY2, TGT2, gapo=4, gape=1, w=50, zdrop=400, impl=impl)
    assert (f["max"], f["max_q"], f["max_t"], f["score"]) == (0, -1, -1, -75)
    assert orc.cigar_str(cig) == "11D3M1D7M6D16M21D18M1I22M1D17M3D1M"


def test_empty_inputs():
    f, cig, ez = orc.ksw2("", "ACGT")
    assert ez.status == 1 and f["n_cigar"] == 0 and f["max_q"] == -1 and f["score"] == orc.Ez().score - 0x40000000


def random_pair(rng):
    mode = int(rng.integers(0, 4))
    if mode == 0:  # call-site A shape: contig vs reference window with one planted indel (src/indelope.nim:221)
        ql = int(rng.integers(20, 700)); base = rng.integers(0, 4, ql + 400).astype(np.uint8)
        q = base[:ql].copy(); t = base[:ql + int(rng.integers(0, 260))].copy()
        pos = int(rng.integers(1, max(2, ql - 1))); L = int(rng.integers(1, 80))
        if rng.random() < 0.5:
            q = np.concatenate([q[:pos], rng.integers(0, 4, L).astype(np.uint8), q[pos:]])
        else:
            q = np.concatenate([q[:pos], q[min(len(q), pos + L):]])
        if len(q) == 0:
            q = base[:5].copy()
        w, z, go = 50, 400, 4
    elif mode == 1:  # call-site B shape: read vs suffix, unbanded (src/indelope.nim:317-318,343-344)
        ql = int(rng.integers(1, 200)); tl = int(rng.integers(1, 900)); base = rng.integers(0, 4, tl + ql).astype(np.uint8)
        o = int(rng.integers(0, tl)); t = base[:tl].copy(); q = base[o:o + ql].copy()
        w, z, go = -1, -1, 5
    elif mode == 2:  # random parameters
        ql = int(rng.integers(1, 400)); tl = int(rng.integers(1, 500)); base = rng.integers(0, 4, max(ql, tl) + 50).astype(np.uint8)
        q = base[:ql].copy(); t = base[:tl].copy()
        w = int(rng.integers(1, 70)); z = int(rng.integers(50, 350)); go = int(rng.integers(1, 7))
    else:  # tandem repeats
        unit = rng.integers(0, 4, int(rng.integers(1, 6))).astype(np.uint8)
        q = np.resize(unit, int(rng.integers(5, 300))).copy(); t = np.resize(unit, int(rng.integers(5, 400))).copy()
        w = int(rng.choice([-1, 50, 20])); z = int(rng.choice([-1, 400, 100])); go = int(rng.choice([4, 5]))
    for a in (q, t):
        m = rng.random(len(a)) < 0.02; a[m] = rng.integers(0, 4, int(m.sum()))
        if rng.random() < 0.3:
            m = rng.random(len(a)) < 0.02; a[m] = 4
    return q, t, go, w, z


@needs_ref
def test_lane_model_equals_compiled_reference_fuzz():
    rng = np.random.default_rng(20171101)
    for it in range(6000):
        q, t, go, w, z = random_pair(rng)
        f1, c1, _ = orc.ksw2(q, t, gapo=go, gape=1, w=w, zdrop=z, impl="ref")
        f2, c2, _ = orc.ksw2(q, t, gapo=go, gape=1, w=w, zdrop=z, impl="lane")
        assert f1 == f2 and c1 == c2, (it, len(q), len(t), go, w, z, f1, f2, orc.cigar_str(c1), orc.cigar_str(c2))


LANE_FUZZ = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ksw2_lane_fuzz.npz")


def lane_fuzz_pairs():
    """the 6 000 pairs of test_lane_model_equals_compiled_reference_fuzz"""
    rng = np.random.default_rng(20171101)
    return [random_pair(rng) for _ in range(6000)]


def pairs_digest(pairs):
    """SHA-256 over every pair's parameters and sequences: the inputs the recorded results belong to"""
    h = hashlib.sha256()
    for q, t, go, w, z in pairs:
        h.update(np.array([len(q), len(t), go, w, z], dtype=np.int64).tobytes() + q.tobytes() + t.tobytes())
    return h.hexdigest()


def test_lane_model_reproduces_its_recorded_fuzz_results():
    """Regression vectors, not the reference's output: tests/golden/ksw2_lane_fuzz.npz holds what the lane model (oracle/ksw2_lane.c)
    computes on the pairs of the fuzz above, recorded with ksw2_lane.c as it has been since that fuzz was written.  Any change to the
    lane model's fields or CIGARs fails here even where the compiled reference is not built; where it is built, the fuzz above
    compares the lane model with the reference itself."""
    pairs = lane_fuzz_pairs()
    g = np.load(LANE_FUZZ)
    assert str(g["made_with"]) == "lane" and str(g["inputs_sha256"]) == pairs_digest(pairs), "the fuzz pairs are not the recorded ones"
    off = np.concatenate([[0], np.cumsum(np.maximum(g["fields"][:, orc.EZ_FIELDS.index("n_cigar")], 0))])
    for it, (q, t, go, w, z) in enumerate(pairs):
        f, c, _ = orc.ksw2(q, t, gapo=go, gape=1, w=w, zdrop=z, impl="lane")
        assert [f[k] for k in orc.EZ_FIELDS] == g["fields"][it].tolist() and list(c) == g["cigar"][off[it]:off[it + 1]].tolist(), (it, f, orc.cigar_str(c))
