"""Crafted BGZF members (tests/deflate_cases.py, written by tests/deflate_writer.py, no zlib) through idl_bam_open on the GPU: every valid
construct as the first member of a file, in the middle and as the last before the EOF marker, carrying real BAM bytes (the bytes of one long
record's bases and qualities, which may be anything), checked against util.parse_bam; ISIZE-0 members and EOF markers in the middle of a
file, extra subfields around BC, members of exactly 64 KiB; and corrupt members, each refused with the decoder's error for the lowest bad
member.  The one-lane CPU build of the same decoder runs the same corpus in tests/test_inflate_crafted.py, under AddressSanitizer too."""
import random
import re

import pytest

from indelope_b200 import cuda
import deflate_cases as dc
import deflate_writer as dw
import idl_testutil as util
from test_gpu_bam import check_against_parse

pytestmark = pytest.mark.gpu

REFS = [("chr1", 5_000_000)]
SMALL = [util.bam_record(0, 10 + k, [("M", 4)], "ACGT", name=b"s%d" % k) for k in range(3)]
ERROR_TEXT = {dc.E_BTYPE: "reserved deflate block type", dc.E_STORED: "stored block length check failed", dc.E_CODE: "invalid Huffman code",
              dc.E_SYMBOL: "invalid symbol", dc.E_DISTANCE: "match distance before the start of the member",
              dc.E_OUTPUT: "inflated size differs from ISIZE", dc.E_INPUT: "compressed data ends early"}


def long_head(n):
    """the bytes of a record in front of its bases and qualities, which are its last n bytes (n a multiple of 3: l / 2 + l)"""
    assert n % 3 == 0
    l = 2 * n // 3
    rec = util.bam_record(0, 1000, [("M", l)], "A" * l, qual=[0] * l, name=b"long")
    return rec[:len(rec) - n]


PREFIX_LEN = len(util.bam_bytes(REFS, SMALL)) + len(long_head(3))


def crafted(builder, seed, head=b"", before=b"", after=b""):
    blocks = builder(random.Random(seed), len(head))
    plan = ([{"type": "stored", "data": head, "final": False}] if head else []) + blocks
    s, p, _ = dw.deflate(plan)
    assert p is not None
    return dw.bgzf_wrap(s, p, before=before, after=after), p[len(head):]


def assemble(pieces, seed=0):
    """pieces: ("crafted", builder[, before, after]) | ("zlib", n random bytes) | ("member", bgzf bytes, payload).  The first piece must be
    crafted: the BAM header and the long record's head go in front of it as a stored block of the same member.  The payloads of all pieces
    are the long record's bases and qualities; the last piece ends the file before the EOF marker."""
    rng = random.Random(seed)
    assert pieces[0][0] == "crafted"
    sizes = []
    for k, pc in enumerate(pieces):
        if pc[0] == "crafted":
            _, p = crafted(pc[1], seed * 1000 + k, head=bytes(PREFIX_LEN) if k == 0 else b"")
            sizes.append(len(p))
        elif pc[0] == "zlib":
            sizes.append(pc[1])
        else:
            sizes.append(len(pc[2]))
    fix = (-sum(sizes)) % 3
    z = [k for k, pc in enumerate(pieces) if pc[0] == "zlib"]
    assert z or not fix
    if fix:
        sizes[z[0]] += fix
    prefix = util.bam_bytes(REFS, SMALL) + long_head(sum(sizes))
    assert len(prefix) == PREFIX_LEN
    members, q = [], []
    for k, pc in enumerate(pieces):
        if pc[0] == "crafted":
            m, p = crafted(pc[1], seed * 1000 + k, head=prefix if k == 0 else b"", before=pc[2] if len(pc) > 2 else b"",
                           after=pc[3] if len(pc) > 3 else b"")
            assert len(p) == sizes[k]
        elif pc[0] == "zlib":
            p = bytes(rng.choice(b"ACGT!#+") for _ in range(sizes[k]))
            m = b"".join(util.bgzf_member(p[i:i + 0xff00]) for i in range(0, len(p), 0xff00))
        else:
            m, p = pc[1], pc[2]
        members.append(m)
        q.append(p)
    raw = prefix + b"".join(q)
    return raw, b"".join(members) + util.BGZF_EOF


def opened(raw, data):
    b, _ = check_against_parse(raw, data)
    assert b.n_records == len(SMALL) + 1 and b.info["inflated_bytes"] == len(raw)
    b.close()


@pytest.mark.parametrize("name", list(dc.VALID))
def test_valid_construct_first_middle_and_last(name):
    build = dc.VALID[name]
    raw, data = assemble([("crafted", build), ("zlib", 30_000), ("crafted", build), ("zlib", 5000), ("crafted", build)], seed=len(name))
    opened(raw, data)


def test_every_short_distance_at_every_length():
    """distances 1-40 at lengths 3-258, one member each: the overlapping copies of the warp (lane i copies byte i mod dist)"""
    pieces = [("crafted", dc.VALID["small_codes"])] + [("crafted", dc.DISTS["dist_%d" % d]) for d in range(1, 41)]
    raw, data = assemble(pieces[:1] + [("zlib", 1000)] + pieces[1:], seed=7)
    opened(raw, data)


def test_empty_members_extra_subfields_and_full_members():
    """ISIZE-0 members and EOF markers in the middle (as `cat a.bam b.bam` leaves them), XLEN > 6 with a subfield before and after BC, and
    members of exactly 65536 bytes"""
    empty = dw.bgzf_wrap(b"\x03\x00", b"")
    sub1, sub2 = dw.subfield(b"XY", b"abc"), dw.subfield(b"RG", b"")
    fp = bytes(range(256)) * 255 + bytes(225)                               # 65505 bytes: a stored block of 65510, a member of 65536
    full = dw.bgzf_wrap(dw.deflate([{"type": "stored", "data": fp}])[0], fp)
    assert len(full) == 65536
    p = bytes(65505 - len(sub1) - len(sub2))
    full_x = dw.bgzf_wrap(dw.deflate([{"type": "stored", "data": p}])[0], p, before=sub1, after=sub2)
    assert len(full_x) == 65536
    pieces = [("crafted", dc.VALID["stored_blocks"], sub1, sub2), ("member", empty, b""), ("member", util.BGZF_EOF, b""), ("zlib", 20_000),
              ("member", empty, b""), ("member", full, fp), ("crafted", dc.VALID["small_codes"], b"", sub1), ("member", full_x, p),
              ("member", util.BGZF_EOF, b""), ("member", empty, b""), ("crafted", dc.VALID["special_matches"], sub2, b"")]
    raw, data = assemble(pieces, seed=9)
    opened(raw, data)


def _good_members(n):
    rng = random.Random(n)
    raw = util.bam_bytes(REFS, SMALL) + bytes(rng.choice(b"ACGT") for _ in range(4000 * n))
    return [util.bgzf_member(raw[i:i + 4000]) for i in range(0, len(raw), 4000)]


def _bad_member(name):
    plan, expect, isize = dc.INVALID[name]
    s, p, F = dw.deflate(plan)
    return dw.bgzf_wrap(s, p or b"", isize=F["out_len"] if isize is None else isize, crc=0), expect


def _refused(data, index, expect):
    texts = "|".join(re.escape(ERROR_TEXT[e]) for e in sorted(expect))
    with pytest.raises(cuda.IdlError, match=r"BGZF block %d failed to inflate \(corrupt data or CRC mismatch: (%s)\)" % (index, texts)):
        cuda.Bam(data)


@pytest.mark.parametrize("name", list(dc.INVALID))
def test_corrupt_member_is_refused(name):
    good = _good_members(6)
    bad, expect = _bad_member(name)
    _refused(b"".join(good[:3] + [bad] + good[3:]) + util.BGZF_EOF, 3, expect)
    if name.startswith("runaway"):                                       # a block that runs off the last member of the file
        _refused(b"".join(good + [bad]) + util.BGZF_EOF, len(good), expect)


def test_the_lowest_bad_member_is_named():
    good = _good_members(12)
    names = ["runaway_15bit", "incomplete_dist", "stored_nlen", "btype_3", "distance_before_start"]
    members = list(good)
    for k, n in zip((11, 9, 7, 5, 4), names):
        members.insert(k, _bad_member(n)[0])
    _refused(b"".join(members) + util.BGZF_EOF, 4, {dc.E_DISTANCE})
