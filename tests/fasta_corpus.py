"""Crafted FASTA texts and their BGZF forms for the bgzipped-reference tests (test_fasta_bgzf_host.py, test_gpu_fasta.py).

The rules are those of the host loader (load_fasta in indelope_b200/csrc/host/bamio.cpp): lines end at '\\n'; a line whose first byte is '>' starts
a record named by the rest of the line up to the first ' ', '\\t' or '\\r'; every other line belongs to the latest record, kept verbatim but for its
trailing run of '\\r' and ' '."""
import gzip
import random
import struct
import zlib

import idl_testutil as util

MEMBER_SIZES = (1, 2, 3, 7, 61, 4096, 0xff00)
# (level, strategy) pairs cycled over the members: stored, fixed-Huffman and dynamic blocks in one file
LEVELS = ((6, zlib.Z_DEFAULT_STRATEGY), (0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_FIXED), (9, zlib.Z_HUFFMAN_ONLY), (4, zlib.Z_RLE))


def wrap(seq, width):
    return b"".join(seq[i:i + width] + b"\n" for i in range(0, len(seq), width))


def parse(text):
    """the loader's rules in Python: [(name, sequence)]; ValueError for a text that does not start with '>'"""
    if text and text[:1] != b">":
        raise ValueError("FASTA record does not start with '>'")
    recs = []
    for line in text.split(b"\n") if text else []:
        if line[:1] == b">":
            name = line[1:]
            for d in (b" ", b"\t", b"\r"):
                name = name.split(d, 1)[0]
            recs.append([name, bytearray()])
        else:
            recs[-1][1] += line.rstrip(b"\r ")
    return [(n.decode("latin-1"), bytes(s)) for n, s in recs]


def corpus():
    """name -> text"""
    rng = random.Random(11)
    acgt = lambda n: bytes(rng.choice(b"ACGT") for _ in range(n))  # noqa: E731
    seq = acgt(1000)
    t = {}
    t["crlf"] = b">c1 desc\r\n" + wrap(seq[:300], 60).replace(b"\n", b"\r\n") + b">c2\r\n" + wrap(seq[300:500], 61).replace(b"\n", b"\r\n")
    t["trailing_spaces"] = b">s1\n" + b"".join(seq[i:i + 50] + b" " * (i % 4) + b"\n" for i in range(0, 400, 50))
    t["mixed_cr_space_runs"] = b">m1\n" + b"".join(seq[i:i + 40] + rng.choice([b" \r", b"\r \r", b"  \r\r ", b"\r", b""]) + b"\n" for i in range(0, 600, 40))
    t["inner_spaces_kept"] = b">i1\nAC GT\r\nA\rC \r\n \r \nG\n"
    t["blank_lines"] = b">b1\n\n" + seq[:70] + b"\n\n\n" + seq[70:90] + b"\n\r\n \n>b2\n\n"
    t["gt_inside_lines"] = b">g1\nACG>T\nA>>\n >G\n>g2 x>y\nTT>\n"
    t["headers"] = b">h1 with spaces\nAC\n>h2\twith tab\nGT\n>h3\rcr\nAA\n>h4\n>h5 \n\n>h6\t\nC\n"
    t["header_only"] = b">lonely description"
    t["no_final_newline"] = b">n1\n" + wrap(seq[:130], 60)[:-1]
    t["empty"] = b""
    t["alphabet"] = b">a1\nacgtnACGTNRYKMSWBDHVN-*.\n" + bytes([0, 1, 2, 9, 11, 12]) + b"\n" + bytes(range(0x80, 0x100)) + b"\n>a2\nacgtacgtNNNNnnnn\n"
    for w in (1, 60, 61, 80):
        t["width_%d" % w] = b">w%d\n" % w + wrap(seq, w) + b">w%d_b\n" % w + wrap(seq[:333], w)
    t["mixed_widths"] = b">mw\n" + b"".join(seq[i:i + k] + b"\n" for i, k in zip(range(0, 1000, 50), [50, 10, 70, 50, 1, 49] * 10)) + b">mw2\n" + seq[:5] + b"\n" + seq[5:200] + b"\n"
    t["duplicate_names"] = b">dup\nAAAA\n>dup second\nCCCC\n>other\nG\n>dup\nTT\n"
    t["many_records"] = b"".join(b">r%d\n" % k + wrap(acgt(k % 97), 13) for k in range(300))
    big = acgt(5_000_000)
    t["unwrapped_5mb"] = b">big\n" + big + b"\n>tail\nACGT\n"
    return t


def large(name):
    """the GPU-only texts: a 50 Mb unwrapped record; a 2 x 40 Mb reference in 60 columns with soft-masked stretches and N runs"""
    rng = random.Random(13)
    if name == "unwrapped_50mb":
        return b">u50 unwrapped\n" + rng.randbytes(50_000_000).translate(bytes(b"ACGT"[i & 3] for i in range(256))) + b"\n"
    out = []
    for c in range(2):
        s = bytearray(rng.randbytes(40_000_000).translate(bytes(b"ACGT"[i & 3] for i in range(256))))
        for _ in range(200):
            a = rng.randrange(0, len(s) - 20000); k = rng.randrange(1, 20000)
            s[a:a + k] = s[a:a + k].lower() if rng.random() < 0.7 else b"N" * k
        out.append(b">chr%d\n" % (c + 1) + wrap(bytes(s), 60))
    return b"".join(out)


def member_sizes(text):
    return MEMBER_SIZES if len(text) < 200_000 else (4096, 0xff00)


def bgzf(text, block, levels=LEVELS):
    return util.bgzf_compress(text, block=block, levels=levels)


def bgzf_cut(text, cuts, level=6):
    """BGZF with a member boundary at every offset in cuts (and every 0xff00 bytes between them)"""
    edges = sorted(set(list(range(0, len(text), 0xff00)) + [c for c in cuts if 0 < c < len(text)] + [len(text)]))
    return b"".join(util.bgzf_member(text[a:b], level) for a, b in zip(edges, edges[1:])) + util.BGZF_EOF


def errors():
    """name -> (bytes, phrase the message must contain)"""
    text = b">e1\n" + b"ACGT" * 5000 + b"\n>e2\nGG\n"
    good = util.bgzf_compress(text, block=4096, level=6)
    out = {}
    out["plain_gzip"] = (gzip.compress(text, 6), "bgzip")
    m0 = util.bgzf_member(text[:4096], 6)
    rest = util.bgzf_compress(text[4096:], block=4096, level=6)
    flipped = bytearray(m0); flipped[30] ^= 0x55
    out["flipped_byte"] = (bytes(flipped) + rest, "failed to inflate")
    bad_crc = bytearray(m0); bad_crc[-8] ^= 1
    out["wrong_crc"] = (bytes(bad_crc) + rest, "failed to inflate")
    bad_isize = bytearray(m0); bad_isize[-4:] = struct.pack("<I", 4095)
    out["wrong_isize"] = (bytes(bad_isize) + rest, "failed to inflate")
    out["truncated_member"] = (good[:len(m0) + 40], "truncated BGZF block")
    out["starts_with_newline"] = (util.bgzf_compress(b"\n" + text), "does not start with '>'")
    out["starts_with_base"] = (util.bgzf_compress(b"A" + text), "does not start with '>'")
    return out
