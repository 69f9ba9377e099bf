"""The crafted DEFLATE corpus shared by tests/test_inflate_crafted.py (the one-lane CPU build) and tests/test_gpu_bam_crafted.py (BGZF
members through idl_bam_open): plans for tests/deflate_writer.py of the constructs zlib's encoder never writes, valid and invalid.

VALID[name](rng, op0) -> list of blocks.  op0 is the number of bytes a block in front of them has already produced in the same member (the
GPU tests put the BAM header there); distances that must reach a given byte take it into account.
INVALID[name] = (plan, expected decoder errors, isize or None for the payload's length)."""
import deflate_writer as dw
from deflate_writer import EOB, LEN_BASE, LEN_EXTRA, DIST_BASE, DIST_EXTRA

# decoder status codes (inflate_core.cuh)
OK, E_BTYPE, E_STORED, E_CODE, E_SYMBOL, E_DISTANCE, E_OUTPUT, E_INPUT = 0, 1, 2, 3, 4, 5, 6, 7
SHORT = [ord(c) for c in "ACGTNacgtn"]


def rbytes(rng, n):
    return bytes(rng.getrandbits(8) for _ in range(n))


def max_len(ls):
    """the longest length symbol ls codes: its largest extra value"""
    return 258 if ls == 285 else LEN_BASE[ls - 257] + (1 << LEN_EXTRA[ls - 257]) - 1


def max_dist(ds):
    return DIST_BASE[ds] + (1 << DIST_EXTRA[ds]) - 1


def lit_every_length(rng, op0=0):
    """literal/length code words of every length 1-15 in one code (a comb 1, 2, ..., 14, 15, 15); then codes that put EOB, all 29 length
    symbols and bytes on 11-15-bit words, and every distance symbol on a 9-15-bit word, each at its largest extra value (distance 32768
    included, behind 33000 stored bytes)"""
    lit = {s: i + 1 for i, s in enumerate(SHORT)}
    lit.update({ord("x"): 11, 257: 12, 285: 13, EOB: 14, ord("y"): 15, 270: 15})
    toks = SHORT + [ord("x"), ord("y")]
    rng.shuffle(toks)
    a = {"type": "dynamic", "lit": lit, "tokens": toks + [(3, 1), (258, 2), (26, 3)]}
    blocks = [a, {"type": "stored", "data": rbytes(rng, 33000)}]
    lsyms = list(range(257, 286))
    for k, (nshort, shape) in enumerate(((10, "balanced"), (9, "comb"))):
        fill = [EOB] + lsyms + [ord("q"), ord("r")] if nshort == 10 else [EOB] + lsyms + [ord("n"), ord("q")]
        rng.shuffle(fill)
        lit = dw.complete({s: i + 1 for i, s in enumerate(SHORT[:nshort])}, fill, 15, shape)
        short_d = list(range(22, 30)) if k == 0 else list(range(8))
        long_d = [d for d in range(30) if d not in short_d]
        rng.shuffle(long_d)
        pin = {d: i + 1 for i, d in enumerate(short_d)}
        if k == 1:
            pin[long_d[0]] = 11                  # (the comb of the other block has no 11-bit word)
        dist = dw.complete(pin, [d for d in long_d if d not in pin], 15, "comb")
        toks = SHORT[:nshort] + [ord("q")]
        for i in range(max(len(lsyms), len(long_d))):
            ls, ds = lsyms[i % len(lsyms)], long_d[i % len(long_d)]
            toks.append(("match", max_len(ls), max_dist(ds), ls))
        blocks.append({"type": "dynamic", "lit": lit, "dist": dist, "tokens": toks, "hclen": 19})
    return blocks


def small_codes(rng, op0=0):
    """a distance code of one 1-bit code word (symbol 0, then symbol 5), a literal-only block with HDIST = 1 and length 0, an empty block
    whose literal code is EOB alone on a 1-bit word; HLIT 257 and 286, HDIST 1 and 30"""
    data = [rng.choice(SHORT) for _ in range(300)]
    return [
        {"type": "dynamic", "tokens": data[:100] + [(10, 1), (258, 1)] + data[100:120] + [(3, 1)], "dist": {0: 1}},
        {"type": "dynamic", "tokens": data[120:200], "dist": {}},                                    # HDIST 1, its length 0
        {"type": "dynamic", "tokens": [], "lit": {EOB: 1}, "dist": {}},
        {"type": "dynamic", "tokens": data[200:260] + [(7, 7), (8, 8), (9, 8)], "dist": {5: 1}},
        {"type": "dynamic", "tokens": data[260:] + [(4, 30)], "hlit": 286, "hdist": 30},
    ]


def code_length_code(rng, op0=0):
    """HCLEN 19 and a code-length code with 7-bit code words (a comb over the symbols the block uses)"""
    data = bytes(rng.choice(b"ACGTNacgtnXYZ0123456789") for _ in range(2000))
    toks = list(data[:40]) + [(40 + k % 50, 1 + k % 30) for k in range(60)] + list(data[40:])
    return [{"type": "dynamic", "tokens": toks, "deep": [ord("9"), ord("Z")],
             "cl_lens": lambda f, lim: dw.complete({}, sorted(f, key=lambda s: (-f[s], s)), lim, "comb"), "hclen": 19}]


def repeats_across(rng, op0=0):
    """code-length repeats 16, 17 and 18 that cross from the literal/length lengths into the distance lengths (one sequence, as libdeflate
    writes it), 16 directly after a 17 or 18 (it repeats a zero), and 18 with 138"""
    filler = bytes(rng.choice(SHORT) for _ in range(4000))
    blocks = [{"type": "stored", "data": filler, "final": False}]
    # 16: lit 280..285 and dist 0..15 all 4 bits long
    lit = dw.complete({s: 4 for s in range(280, 286)}, SHORT[:4] + [EOB], 15)
    blocks.append({"type": "dynamic", "lit": lit, "dist": {d: 4 for d in range(16)}, "cl": "joint",
                   "tokens": [rng.choice(SHORT[:4]) for _ in range(50)] + [(258, 1), (131, 4), (163, 9), (195, 200), (227, 150)]})
    # 17: lit 283..285 and dist 0..2 zero (6 zeros); 18: lit 276..285 and dist 0..4 zero (15 zeros)
    for last_lit, first_dist in ((282, 3), (275, 5)):
        lit = dw.complete({}, SHORT[:4] + [EOB, 257, last_lit], 15)
        dist = dw.complete({}, list(range(first_dist, first_dist + 4)), 15)
        toks = [rng.choice(SHORT[:4]) for _ in range(60)]
        toks += [("match", 3, max_dist(d), 257) for d in dist] + [("match", max_len(last_lit), DIST_BASE[first_dist], last_lit)]
        blocks.append({"type": "dynamic", "lit": lit, "dist": dist, "hlit": 286, "cl": "joint", "tokens": toks})
    # 16 after 17 / 18, and 18 with 138: bytes 0..199 unused (a zero run of 200)
    hi = list(range(200, 256))
    lit = dw.complete({}, hi + [EOB, 257, 258], 15)
    seq = [lit.get(s, 0) for s in range(259)] + [1, 1]
    items = []
    for s, x in dw.rle_lengths(seq, "joint", 259):
        if s == 18 and 3 <= x < 127:
            items += [(18, x - 3), (16, 0)]        # the same zeros, the last three as a repeat of the zero before them
        elif s == 17 and x >= 3:
            items += [(17, x - 3), (16, 0)]
        else:
            items.append((s, x))
    toks = [rng.choice(hi) for _ in range(300)] + [(3, 1), (4, 2), (3, 2)]
    blocks.append({"type": "dynamic", "lit": lit, "dist": {0: 1, 1: 1}, "hlit": 259, "hdist": 2, "cl": items, "tokens": toks})
    # 16 after a 17 that crosses into the distance lengths: lit 258, 259 and dist 0 by the 17, dist 1..3 by the 16
    lit = dw.complete({}, SHORT[:4] + [EOB, 257], 15)
    items = dw.rle_lengths([lit.get(s, 0) for s in range(258)], "joint", 258) + [(17, 0), (16, 0), (0, 0), (0, 0), (1, 0), (1, 0)]
    toks = [rng.choice(SHORT[:4]) for _ in range(300)] + [(3, 9), (3, 13)]
    blocks.append({"type": "dynamic", "lit": lit, "dist": {6: 1, 7: 1}, "hlit": 260, "hdist": 8, "cl": items, "tokens": toks})
    return blocks


def stored_blocks(rng, op0=0):
    """stored LEN 0 (non-final and final), a stored header at each of the 8 bit phases (a fixed block of 0-7 nine-bit literals in front), and
    stored data that starts at every offset modulo 128 (129-byte steps)"""
    blocks = [{"type": "stored", "data": b""}]
    for j in range(8):
        blocks.append({"type": "fixed", "tokens": [rng.choice(SHORT) for _ in range(5)] + [200 + k for k in range(j)]})
        blocks.append({"type": "stored", "data": rbytes(rng, rng.choice([1, 31, 32, 33, 300]))})
    for i in range(128):
        blocks.append({"type": "stored", "data": rbytes(rng, 124)})
    blocks.append({"type": "stored", "data": b"", "final": True})
    return blocks


def dist_all_lengths(d):
    """distance d at every length 3-258 (overlapping copies where d < length: on the device lane i copies byte i mod d)"""
    def build(rng, op0=0):
        toks = list(rbytes(rng, 40)) + [(length, d) for length in range(3, 259)]
        return [{"type": "fixed" if d % 2 else "dynamic", "tokens": toks}]
    return build


def special_matches(rng, op0=0):
    """a distance back to the first byte of the member (dist == op), distances 2047/2048/2049 (the decoder's ring), 32768, and length 258 as
    285 and as 284 + 31"""
    toks = list(rbytes(rng, 100))
    toks += [(3, op0 + 100), (258, op0 + 103)]                              # to the member's first byte
    toks += list(rbytes(rng, 2000)) + [(l, d) for d in (2047, 2048, 2049) for l in (3, 31, 32, 33, 258)]
    toks += [("match", 258, 2048, 284), ("match", 258, 2049, 285), ("match", 258, 100, 284)]
    toks2 = list(rbytes(rng, 12000))
    return [{"type": "dynamic", "tokens": toks}, {"type": "stored", "data": rbytes(rng, 20000)},
            {"type": "fixed", "tokens": toks2 + [(258, 32768), (3, 32768), ("match", 258, 32768, 284)]}]


def many_empty_blocks(rng, op0=0):
    """1001 empty fixed blocks in front of the data, then block types alternating within the member"""
    data = [rng.choice(SHORT) for _ in range(3000)]
    blocks = [{"type": "fixed", "tokens": []} for _ in range(1001)]
    for k in range(12):
        part = data[k * 250:(k + 1) * 250]
        t = ("stored", "fixed", "dynamic")[k % 3]
        blocks.append({"type": t, "data": bytes(part)} if t == "stored" else {"type": t, "tokens": part[:100] + [(20, 7)] + part[100:]})
    return blocks


VALID = {
    "lit_every_length": lit_every_length,
    "small_codes": small_codes,
    "code_length_code": code_length_code,
    "repeats_across": repeats_across,
    "stored_blocks": stored_blocks,
    "special_matches": special_matches,
    "many_empty_blocks": many_empty_blocks,
}
DISTS = {"dist_%d" % d: dist_all_lengths(d) for d in range(1, 41)}


def stored_65535(rng, isize):
    """LEN 65535 in a member of ISIZE 65535 or 65536 (too large for a BGZF member with its framing: CPU only)"""
    blocks = [{"type": "stored", "data": rbytes(rng, 65535)}]
    return ([{"type": "fixed", "tokens": [65]}] if isize == 65536 else []) + blocks


def _lit_code(extra=()):
    return dw.complete({}, SHORT[:4] + [EOB] + list(extra), 15)


def _over_cl(f, lim):
    return {s: 1 for s in f}


def _incomplete_cl(f, lim):
    return {s: 5 for s in f}


def _runaway_comb():
    lit = {s: i + 1 for i, s in enumerate(SHORT)}
    lit.update({ord("x"): 11, 257: 12, 285: 13, EOB: 14, ord("y"): 15, 270: 15})
    return lit


def _bad_repeat_items():
    lit = _lit_code()
    seq = [lit.get(s, 0) for s in range(257)] + [1, 1, 0, 0, 0]
    items = dw.rle_lengths(seq, "joint", 257)
    assert items[-1] == (17, 0)
    return lit, items[:-1] + [(17, 3)]


def _invalid():
    lit2 = _lit_code([257])
    lit_b, items_b = _bad_repeat_items()
    toks = [65, 67, 71, 84] * 10
    return {
        # incomplete codes other than the empty and the single-1-bit ones
        "incomplete_lit": ([{"type": "dynamic", "lit": {65: 2, 66: 2, EOB: 2}, "tokens": [65, 66]}], {E_CODE}, None),
        "incomplete_lit_single_2bit": ([{"type": "dynamic", "lit": {EOB: 2}, "tokens": []}], {E_CODE}, None),
        "incomplete_dist": ([{"type": "dynamic", "lit": lit2, "dist": {0: 2, 1: 2}, "tokens": toks + [(3, 1)]}], {E_CODE}, None),
        "incomplete_dist_single_2bit": ([{"type": "dynamic", "lit": lit2, "dist": {0: 2}, "tokens": toks + [(3, 1)]}], {E_CODE}, None),
        "incomplete_cl": ([{"type": "dynamic", "tokens": toks, "cl_lens": _incomplete_cl}], {E_CODE}, None),
        "incomplete_cl_single_1bit": ([{"type": "dynamic", "lit": {s: 9 for s in range(257)}, "dist": {0: 9}, "tokens": [],
                                        "cl": [(9, 0)] * 258, "cl_lens": {9: 1}}], {E_CODE}, 0),
        # over-subscribed
        "over_lit": ([{"type": "dynamic", "lit": {65: 1, 66: 1, EOB: 1}, "tokens": [65, 66]}], {E_CODE}, None),
        "over_dist": ([{"type": "dynamic", "lit": lit2, "dist": {0: 1, 1: 1, 2: 1}, "tokens": toks + [(3, 1)]}], {E_CODE}, None),
        "over_cl": ([{"type": "dynamic", "tokens": toks, "cl_lens": _over_cl}], {E_CODE}, None),
        # header counts and repeats
        "hlit_287": ([{"type": "dynamic", "tokens": toks, "hlit": 287}], {E_CODE}, None),
        "hlit_288": ([{"type": "dynamic", "tokens": toks, "hlit": 288}], {E_CODE}, None),
        "hdist_31": ([{"type": "dynamic", "tokens": toks + [(3, 1)], "hdist": 31}], {E_CODE}, None),
        "hdist_32": ([{"type": "dynamic", "tokens": toks + [(3, 1)], "hdist": 32}], {E_CODE}, None),
        "repeat_16_first": ([{"type": "dynamic", "lit": lit2, "dist": {0: 1}, "tokens": toks,
                              "cl": [(16, 0)] + dw.rle_lengths([lit2.get(s, 0) for s in range(258)] + [1], "joint", 258)}], {E_CODE}, None),
        "repeat_past_end": ([{"type": "dynamic", "lit": lit_b, "dist": {0: 1, 1: 1}, "hdist": 5, "cl": items_b, "tokens": toks}], {E_CODE}, None),
        "eob_length_0": ([{"type": "dynamic", "lit": {65: 1, 66: 1}, "dist": {}, "tokens": [65], "eob": False}], {E_CODE}, None),
        "hclen_4_no_eob": ([{"type": "dynamic", "lit": {}, "dist": {}, "tokens": [], "eob": False}], {E_CODE}, 0),
        # symbols
        "fixed_lit_286": ([{"type": "fixed", "tokens": toks + [("raw", 286, None)]}], {E_SYMBOL}, 41),
        "fixed_lit_287": ([{"type": "fixed", "tokens": toks + [("raw", 287, None)]}], {E_SYMBOL}, 41),
        "fixed_dist_30": ([{"type": "fixed", "tokens": toks + [("raw", 257, 30)]}], {E_SYMBOL}, 43),
        "fixed_dist_31": ([{"type": "fixed", "tokens": toks + [("raw", 257, 31)]}], {E_SYMBOL}, 43),
        "dynamic_dist_empty_used": ([{"type": "dynamic", "lit": lit2, "dist": {}, "tokens": toks + [("raw", 257, "bits", (0, 1))]}], {E_SYMBOL}, 43),
        "dynamic_dist_single_other_half": ([{"type": "dynamic", "lit": lit2, "dist": {0: 1}, "tokens": toks + [("raw", 257, "bits", (1, 1))]}],
                                           {E_SYMBOL}, 43),
        # distances, stored blocks, sizes, block type
        "distance_before_start": ([{"type": "fixed", "tokens": [65, (3, 2)]}], {E_DISTANCE}, 4),
        "distance_one_too_far": ([{"type": "dynamic", "tokens": toks + [(10, 41)]}], {E_DISTANCE}, 50),
        "stored_nlen": ([{"type": "stored", "data": b"abc", "nlen": 0x1234}], {E_STORED}, None),
        "stored_past_end": ([{"type": "stored", "data": b"x" * 50, "len": 100}], {E_INPUT}, 100),
        "stored_past_end_after_fixed": ([{"type": "fixed", "tokens": toks}, {"type": "stored", "data": b"x" * 7, "len": 8}], {E_INPUT}, 48),
        "isize_short": ([{"type": "fixed", "tokens": toks}], {E_OUTPUT}, 39),
        "isize_long": ([{"type": "fixed", "tokens": toks}], {E_OUTPUT}, 41),
        "isize_short_stored": ([{"type": "stored", "data": b"y" * 300}], {E_OUTPUT}, 299),
        "isize_short_match": ([{"type": "dynamic", "tokens": toks + [(258, 4)]}], {E_OUTPUT}, 100),
        "btype_3": ([{"type": "reserved"}], {E_BTYPE}, 0),
        "btype_3_after_fixed": ([{"type": "fixed", "tokens": toks, "final": False}, {"type": "reserved"}], {E_BTYPE}, 40),
        # a block without an end-of-block that runs off the member
        "runaway_1bit": ([{"type": "dynamic", "lit": {65: 1, EOB: 1}, "dist": {}, "tokens": [65] * 20, "eob": False}], {E_INPUT, E_OUTPUT}, 65536),
        "runaway_fixed": ([{"type": "fixed", "tokens": toks, "eob": False}], {E_INPUT, E_OUTPUT}, 65536),
        "runaway_8bit": ([{"type": "dynamic", "lit": dw.complete({}, list(range(256)) + [EOB, 257], 15), "dist": {0: 1}, "tokens": toks,
                           "eob": False}], {E_INPUT, E_OUTPUT}, 65536),
        "runaway_15bit": ([{"type": "dynamic", "lit": _runaway_comb(), "dist": {0: 1}, "tokens": [ord("y")] * 4000, "eob": False}],
                          {E_INPUT, E_OUTPUT}, 65536),
        "runaway_after_stored": ([{"type": "stored", "data": b"z" * 3000, "final": False},
                                  {"type": "dynamic", "lit": {65: 1, EOB: 1}, "dist": {}, "tokens": [65] * 9, "eob": False}], {E_INPUT, E_OUTPUT}, 65536),
    }


INVALID = _invalid()
