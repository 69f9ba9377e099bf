"""A DEFLATE (RFC 1951) writer for tests: turns an explicit PLAN into a raw deflate stream and reports what the stream really contains.

Written from the RFC, with no zlib inside, so that the decoder's tests reach the parts of the format zlib's encoder never writes: code words of
11-15 bits, single-code and empty distance alphabets, code-length repeats that cross from the literal/length lengths into the distance
lengths (libdeflate writes both as one sequence), 16 right after a run of zeros, stored blocks at any bit phase, and invalid streams of
every kind.

A plan is a list of blocks (dicts):
  {"type": "stored", "data": b"...", "len": LEN override, "nlen": NLEN override}
  {"type": "fixed", "tokens": [...], "eob": True}
  {"type": "dynamic", "tokens": [...], "eob": True,
   "lit": {sym: len} (default: from the frequencies), "dist": {sym: len} (same), "deep": [syms pushed to 15 bits when lengths come from frequencies],
   "hlit": n, "hdist": n (default: the fewest that hold every nonzero length), "cl": "joint" | "split" | [(sym, extra), ...],
   "cl_lens": {sym: len} or f(freq, 7) -> {sym: len} (default: huffman, at most 7 bits), "hclen": n (default: the fewest)}
  {"type": "reserved"}                          BTYPE 3
Every block may carry "final"; by default only the last block is final.
Tokens: an int (a literal byte), (length, distance), ("match", length, distance, length_symbol) to code a length with a chosen symbol
(258 as 284 + 31), or ("raw", lsym, dsym) for a bare literal/length symbol (and distance symbol) with zero extra bits -- how the invalid
symbols 286/287 and distances 30/31 of a fixed block are written; ("raw", lsym, "bits", (value, n)) puts n raw bits where the distance
code word would be.

deflate(plan) -> (stream bytes, payload bytes, feature record); the payload is what a correct decoder outputs (None where a match reaches in
front of the start).  bgzf_wrap() makes a BGZF member of a stream."""
import binascii
import heapq
import struct

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289,
             16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = {s: 8 if s < 144 else 9 if s < 256 else 7 if s < 280 else 8 for s in range(288)}
FIXED_DIST = {s: 5 for s in range(32)}
EOB = 256


class BitWriter:
    """bits go out least significant first (RFC 1951 3.1.1)"""

    def __init__(self):
        self.out, self.acc, self.nacc = bytearray(), 0, 0

    @property
    def pos(self):
        return len(self.out) * 8 + self.nacc

    def bits(self, v, n):
        assert 0 <= v < (1 << n) or n == 0 and v == 0, (v, n)
        self.acc |= v << self.nacc
        self.nacc += n
        while self.nacc >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.nacc -= 8

    def code(self, c, n):
        """a Huffman code word: its most significant bit first (an over-subscribed code's words are cut to n bits)"""
        self.bits(int(format(c & ((1 << n) - 1), "0%db" % n)[::-1], 2) if n else 0, n)

    def align(self):
        if self.nacc:
            self.bits(0, 8 - self.nacc)

    def raw(self, data):
        assert self.nacc == 0
        self.out += data

    def getvalue(self):
        return bytes(self.out) + (bytes([self.acc]) if self.nacc else b"")


def kraft(lens, limit=15):
    """sum of 2^-len in units of 2^-limit; a complete code gives 2^limit"""
    return sum(1 << (limit - l) for l in lens.values() if l)


def canonical(lens):
    """{sym: len} -> {sym: code} (RFC 1951 3.2.2)"""
    count = [0] * 16
    for l in lens.values():
        if l:
            count[l] += 1
    nxt, code = [0] * 16, 0
    for l in range(1, 16):
        code = (code + count[l - 1]) << 1 if l > 1 else 0
        nxt[l] = code
    out = {}
    for s in sorted(lens):
        if lens[s]:
            out[s] = nxt[lens[s]]
            nxt[lens[s]] += 1
    return out


def complete(pinned, fillers, limit=15, shape="balanced"):
    """lengths for `fillers` (in order: the first get the shortest code words) that make {pinned + fillers} a complete code.  The space the
    pinned lengths leave is cut into one piece per filler: "balanced" halves the largest piece, "comb" the smallest that can still be halved
    (a chain of ever longer code words)."""
    left = (1 << limit) - kraft(pinned, limit)
    assert left >= 0, "over-subscribed"
    pieces = [limit - b for b in range(limit + 1) if left >> b & 1]    # lengths, from the binary digits of what is left
    while len(pieces) < len(fillers):
        cand = [l for l in pieces if l < limit]
        assert cand, "too many fillers"
        l = min(cand) if shape == "balanced" else max(cand)
        pieces.remove(l)
        pieces += [l + 1, l + 1]
    assert len(pieces) == len(fillers), "too few fillers for a complete code"
    out = dict(pinned)
    out.update(zip(fillers, sorted(pieces)))
    assert kraft(out, limit) == 1 << limit
    return out


def huffman(freq, limit=15, deep=()):
    """{sym: count} -> {sym: len}, a complete code; the symbols of `deep` (used ones) are pushed to `limit` bits, the others re-fitted by
    frequency, so the Kraft sum stays exact"""
    syms = [s for s in freq if freq[s]]
    if len(syms) == 1:
        return {syms[0]: 1, (syms[0] + 1) % 19 if limit == 7 else syms[0] ^ 1: 1}   # two 1-bit code words: complete
    order = sorted(syms, key=lambda s: (-freq[s], s))
    if not deep:
        h = [(freq[s], k, [s]) for k, s in enumerate(order)]
        heapq.heapify(h)
        depth = dict.fromkeys(syms, 0)
        k = len(h)
        while len(h) > 1:
            a, b = heapq.heappop(h), heapq.heappop(h)
            for s in a[2] + b[2]:
                depth[s] += 1
            heapq.heappush(h, (a[0] + b[0], k, a[2] + b[2]))
            k += 1
        if max(depth.values()) <= limit:
            return depth
    pinned = {s: limit for s in deep}
    return complete(pinned, [s for s in order if s not in pinned], limit)


def len_symbol(length):
    if length == 258:
        return 285
    i = max(k for k in range(28) if LEN_BASE[k] <= length)
    return 257 + i


def dist_symbol(dist):
    return max(k for k in range(30) if DIST_BASE[k] <= dist)


def _symbols(tok):
    """token -> (lsym, lextra, lbits, dsym, dextra, dbits, length, dist)"""
    if isinstance(tok, int):
        return tok, 0, 0, None, 0, 0, 0, 0
    if tok[0] == "raw":
        return tok[1], 0, 0, tok[2:] if tok[2] == "bits" else tok[2], 0, 0, None, None
    if tok[0] == "match":
        _, length, dist, ls = tok
    else:
        length, dist = tok
        ls = len_symbol(length)
    lb = LEN_EXTRA[ls - 257]
    assert LEN_BASE[ls - 257] <= length < LEN_BASE[ls - 257] + (1 << lb) or ls == 285 and length == 258, (length, ls)
    ds = dist_symbol(dist)
    db = DIST_EXTRA[ds]
    assert 1 <= dist <= 32768
    return ls, length - LEN_BASE[ls - 257], lb, ds, dist - DIST_BASE[ds], db, length, dist


def rle_lengths(seq, mode, hlit):
    """code lengths -> [(cl symbol, extra value)]; mode "joint" runs over both alphabets as one sequence, "split" stops every run at hlit"""
    parts = [seq] if mode == "joint" else [seq[:hlit], seq[hlit:]]
    out = []
    for part in parts:
        i = 0
        while i < len(part):
            v, c = part[i], 1
            while i + c < len(part) and part[i + c] == v:
                c += 1
            i += c
            if v == 0:
                while c >= 11:
                    r = min(c, 138)
                    out.append((18, r - 11))
                    c -= r
                if c >= 3:
                    out.append((17, c - 3))
                    c = 0
                out += [(0, 0)] * c
            else:
                out.append((v, 0))
                c -= 1
                while c >= 3:
                    r = min(c, 6)
                    out.append((16, r - 3))
                    c -= r
                out += [(v, 0)] * c
    return out


CL_EXTRA = {16: (2, 3), 17: (3, 3), 18: (7, 11)}   # extra bits, base


def _new_features():
    return dict(blocks=[], lit_lens_used=set(), dist_lens_used=set(), cl_lens_used=set(), lit_long=set(), dist_long_max_extra=set(),
                len_sym_max_extra=set(), hlit=set(), hdist=set(), hclen=set(), cross=set(), rep16_after_zero=False, rep18_138=False,
                stored_phases=set(), stored_data_at=[], stored_lens=[], dists=set(), lens=set(), len_syms=set(), dist_eq_op=False,
                single_dist_code=False, empty_dist_code=False, eob_only_code=False, n_empty_blocks=0, out_len=0)


def deflate(plan):
    bw, F = BitWriter(), _new_features()
    out = bytearray()
    valid = True
    for k, blk in enumerate(plan):
        t = blk["type"]
        final = blk.get("final", k == len(plan) - 1)
        F["blocks"].append(t)
        if t == "stored":
            F["stored_phases"].add(bw.pos % 8)
        bw.bits(int(final), 1)
        bw.bits({"stored": 0, "fixed": 1, "dynamic": 2, "reserved": 3}[t], 2)
        if t == "reserved":
            continue
        if t == "stored":
            data = blk.get("data", b"")
            bw.align()
            ln = blk.get("len", len(data))
            bw.raw(struct.pack("<HH", ln, blk.get("nlen", ln ^ 0xffff)))
            F["stored_data_at"].append(len(bw.out))
            F["stored_lens"].append(len(data))
            bw.raw(data)
            out += data
            F["n_empty_blocks"] += not data
            continue
        toks = [_symbols(tk) for tk in blk.get("tokens", [])]
        if t == "fixed":
            lit, dist = FIXED_LIT, FIXED_DIST
        else:
            lf, df = {}, {}
            for ls, _, _, ds, _, _, _, _ in toks:
                lf[ls] = lf.get(ls, 0) + 1
                if ds is not None:
                    df[ds] = df.get(ds, 0) + 1
            if blk.get("eob", True):
                lf[EOB] = lf.get(EOB, 0) + 1
            lit = blk["lit"] if "lit" in blk else huffman(lf, 15, [s for s in blk.get("deep", ()) if s in lf])
            dist = blk["dist"] if "dist" in blk else huffman(df, 15, [s for s in blk.get("deep", ()) if s in df]) if df else {}
            hlit = blk.get("hlit", max(257, max((s + 1 for s, l in lit.items() if l), default=257)))
            hdist = blk.get("hdist", max(1, max((s + 1 for s, l in dist.items() if l), default=1)))
            seq = [lit.get(s, 0) for s in range(hlit)] + [dist.get(s, 0) for s in range(hdist)]
            cl = blk.get("cl", "joint")
            items = rle_lengths(seq, cl, hlit) if isinstance(cl, str) else list(cl)
            cf = {}
            for s, _ in items:
                cf[s] = cf.get(s, 0) + 1
            cl_lens = blk.get("cl_lens", huffman)
            cl_lens = cl_lens(cf, 7) if callable(cl_lens) else cl_lens
            hclen = blk.get("hclen", max(4, max((i + 1 for i, s in enumerate(CL_ORDER) if cl_lens.get(s, 0)), default=4)))
            bw.bits(hlit - 257, 5)
            bw.bits(hdist - 1, 5)
            bw.bits(hclen - 4, 4)
            for i in range(hclen):
                bw.bits(cl_lens.get(CL_ORDER[i], 0), 3)
            F["hlit"].add(hlit)
            F["hdist"].add(hdist)
            F["hclen"].add(hclen)
            ccodes = canonical(cl_lens)
            n, prev_sym = 0, None
            for s, x in items:
                bw.code(ccodes[s], cl_lens[s])
                F["cl_lens_used"].add(cl_lens[s])
                rep = 1
                if s in CL_EXTRA:
                    nb, base = CL_EXTRA[s]
                    bw.bits(x, nb)
                    rep = base + x
                    if n < hlit < n + rep:
                        F["cross"].add(s)
                    if s == 16 and prev_sym in (17, 18):
                        F["rep16_after_zero"] = True
                    if s == 18 and rep == 138:
                        F["rep18_138"] = True
                n += rep
                prev_sym = s
            used_d = [s for s, l in dist.items() if l]
            if len(used_d) == 1 and dist[used_d[0]] == 1:
                F["single_dist_code"] = True
            if not used_d:
                F["empty_dist_code"] = True
            if [s for s, l in lit.items() if l] == [EOB] and lit[EOB] == 1:
                F["eob_only_code"] = True
        lcodes, dcodes = canonical(lit), canonical(dist)
        for ls, lx, lb, ds, dx, db, length, d in toks:
            bw.code(lcodes[ls], lit[ls])
            F["lit_lens_used"].add(lit[ls])
            if lit[ls] >= 11:
                F["lit_long"].add(ls)
            if ds is None:
                if ls < 256:
                    out.append(ls)
                else:
                    valid = False
                continue
            bw.bits(lx, lb)
            if isinstance(ds, tuple):                 # ("bits", (value, n)): a bit pattern in place of a distance code word
                bw.bits(*ds[1])
                valid = False
                continue
            bw.code(dcodes[ds], dist[ds])
            bw.bits(dx, db)
            F["dist_lens_used"].add(dist[ds])
            if length is None:
                valid = False
                continue
            if lx == (1 << lb) - 1:
                F["len_sym_max_extra"].add((ls, lit[ls]))
            if db == 0 or dx == (1 << db) - 1:
                F["dist_long_max_extra"].add((ds, dist[ds]))
            F["len_syms"].add((ls, lx))
            F["dists"].add(d)
            F["lens"].add(length)
            F["dist_eq_op"] |= d == len(out)
            if d > len(out):
                valid = False
                out += bytes(length)
            else:
                for i in range(length):
                    out.append(out[-d])
        if blk.get("eob", True):
            bw.code(lcodes[EOB], lit[EOB])
            F["lit_lens_used"].add(lit[EOB])
            if lit[EOB] >= 11:
                F["lit_long"].add(EOB)
        if not toks:
            F["n_empty_blocks"] += 1
    F["out_len"] = len(out)
    return bw.getvalue(), bytes(out) if valid else None, F


def subfield(si, data):
    return si + struct.pack("<H", len(data)) + data


def bgzf_wrap(stream, payload, isize=None, crc=None, before=b"", after=b""):
    """a BGZF member (SAM spec 4.1) around a raw deflate stream; CRC and ISIZE default to the payload's, `before` / `after` are extra
    subfields on either side of BC"""
    xlen = len(before) + 6 + len(after)
    bsize = 12 + xlen + len(stream) + 8 - 1
    assert bsize < 65536
    head = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", xlen) + before + b"BC\x02\0" + struct.pack("<H", bsize) + after
    crc = binascii.crc32(payload) if crc is None else crc
    return head + stream + struct.pack("<II", crc, len(payload) if isize is None else isize)
