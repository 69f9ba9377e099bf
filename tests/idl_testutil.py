"""helpers shared by the parity tests"""
import os

import numpy as np

from indelope_b200 import host

HAS_GPU = None


def has_gpu():
    global HAS_GPU
    if HAS_GPU is None:
        try:
            import torch
            HAS_GPU = bool(torch.cuda.is_available())
        except Exception:
            HAS_GPU = False
    return HAS_GPU


def small_dataset(name="pr1", **over):
    cfg = dict(host.CONFIGS[name])
    cfg.update(over)
    return host.Dataset(**cfg)


def diff_lines(a, b, limit=12):
    """first differing lines of two dumps, grouped by record type"""
    la, lb = a.splitlines(), b.splitlines()
    out = []
    if len(la) != len(lb):
        out.append("line counts differ: %d vs %d" % (len(la), len(lb)))
    n = 0
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            out.append("line %d:\n  oracle: %s\n  gpu   : %s" % (i, x[:600], y[:600]))
            n += 1
            if n >= limit:
                break
    return "\n".join(out)


def by_type(dump):
    d = {}
    for l in dump.splitlines():
        d.setdefault(l[:1], []).append(l)
    return d


def rois_from_reads(reads, chrom_seq, roi_start=None, roi_stop=None, chrom_name="chrT"):
    """build a one-region Rois from a list of dicts(start, seq, qual=None, mapq=60, flag=0, stop=None)"""
    starts, stops, mapq, flag, lens, offs = [], [], [], [], [], []
    bases, quals = [], []
    off = 0
    for r in reads:
        s = r["seq"]
        starts.append(r["start"]); stops.append(r.get("stop", r["start"] + len(s))); mapq.append(r.get("mapq", 60)); flag.append(r.get("flag", 0))
        lens.append(len(s)); offs.append(off); off += len(s)
        bases.append(np.frombuffer(s.encode(), dtype=np.uint8))
        q = r.get("qual")
        quals.append(np.full(len(s), 30, dtype=np.uint8) if q is None else np.asarray(q, dtype=np.uint8))
    n = len(reads)
    arrays = dict(
        start=np.array(starts, np.int32), stop=np.array(stops, np.int32), mapq=np.array(mapq, np.uint8), flag=np.array(flag, np.uint16),
        len=np.array(lens, np.int32), seq_off=np.array(offs, np.int64),
        bases=np.concatenate(bases) if bases else np.zeros(0, np.uint8), quals=np.concatenate(quals) if quals else np.zeros(0, np.uint8),
        roi_chrom=np.zeros(1, np.int32), roi_start=np.array([roi_start if roi_start is not None else min(starts)], np.int32),
        roi_stop=np.array([roi_stop if roi_stop is not None else max(stops)], np.int32), roi_read_begin=np.zeros(1, np.int64),
        roi_n_reads=np.array([n], np.int32), read_idx=np.arange(n, dtype=np.int64),
        chrom_names=[chrom_name], chrom_seqs=[np.frombuffer(chrom_seq.encode(), dtype=np.uint8) if isinstance(chrom_seq, str) else chrom_seq],
    )
    return host.Rois(arrays=arrays), arrays


def merge_rois(list_of_arrays, chroms=None, chrom_names=None, chrom_seqs=None):
    """concatenate several one-chromosome region sets into one.  Without `chroms` they share the first set's chromosome; with it,
    set k lies on chromosome chroms[k] of chrom_names / chrom_seqs"""
    out = {k: [] for k in ("start", "stop", "mapq", "flag", "len", "seq_off", "bases", "quals", "roi_chrom", "roi_start", "roi_stop", "roi_read_begin",
                           "roi_n_reads", "read_idx")}
    nread = nbase = nidx = 0
    for j, a in enumerate(list_of_arrays):
        for k in ("start", "stop", "mapq", "flag", "len", "bases", "quals", "roi_start", "roi_stop", "roi_n_reads"):
            out[k].append(a[k])
        out["roi_chrom"].append(a["roi_chrom"] if chroms is None else np.full(len(a["roi_chrom"]), chroms[j], np.int32))
        out["seq_off"].append(a["seq_off"] + nbase)
        out["roi_read_begin"].append(a["roi_read_begin"] + nidx)
        out["read_idx"].append(a["read_idx"] + nread)
        nread += len(a["start"]); nbase += len(a["bases"]); nidx += len(a["read_idx"])
    m = {k: np.concatenate(v) for k, v in out.items()}
    if chroms is None:
        m["chrom_names"] = list_of_arrays[0]["chrom_names"]; m["chrom_seqs"] = list_of_arrays[0]["chrom_seqs"]
    else:
        m["chrom_names"] = list(chrom_names)
        m["chrom_seqs"] = [np.frombuffer(s.encode(), dtype=np.uint8) if isinstance(s, str) else s for s in chrom_seqs]
    return m


# ---------------------------------------------------------------------------------------------------------------
# Directed regions at chromosome ends: reads of a haplotype (reference + edits, with soft-clipped bases in front of the chromosome
# start or past its end), each with its CIGAR, so that one set of reads makes both the Rois arrays and a BAM file
# ---------------------------------------------------------------------------------------------------------------
def random_seq(rng, n, alphabet="ACGT"):
    return "".join(alphabet[i] for i in rng.integers(0, len(alphabet), n))


def haplotype(ref, edits=(), lead="", tail=""):
    """per-base list of (base, reference position or None, kind in M/I/S).  edits: (pos, "I", seq) inserts seq before ref[pos];
    (pos, "D", n) deletes ref[pos:pos + n].  lead / tail: bases before position 0 / after the chromosome's end (soft clips)"""
    ed = {p: (k, a) for p, k, a in edits}
    out = [(c, None, "S") for c in lead]
    i = 0
    while i < len(ref):
        k, a = ed.get(i, (None, None))
        if k == "D":
            i += a
            continue
        if k == "I":
            out += [(c, None, "I") for c in a]
        out.append((ref[i], i, "M"))
        i += 1
    return out + [(c, None, "S") for c in tail]


def hap_read(hp, at, n, qual=None, mapq=60, flag=0):
    """the read of bases [at, at + n) of a haplotype: dict(start, stop, seq, qual, mapq, flag, cigar) as rois_from_reads and
    bam_record take them; insertions at either end of the read become soft clips"""
    seg = hp[at:at + n]
    m = [i for i, (_, p, _) in enumerate(seg) if p is not None]
    assert m, "a read needs an aligned base"
    cig, prev = [], None
    for i, (_, p, k) in enumerate(seg):
        if k == "I" and (i < m[0] or i > m[-1]):
            k = "S"
        if p is not None and prev is not None and p > prev + 1:
            cig.append(["D", p - prev - 1])
        if cig and cig[-1][0] == k:
            cig[-1][1] += 1
        else:
            cig.append([k, 1])
        if p is not None:
            prev = p
    seq = "".join(b for b, _, _ in seg)
    return dict(start=seg[m[0]][1], stop=prev + 1, seq=seq, qual=[30] * len(seq) if qual is None else list(qual), mapq=mapq, flag=flag,
                cigar=[(k, ln) for k, ln in cig])


def _lowq(n, lead=0, trail=0):
    return [4] * lead + [30] * (n - lead - trail) + [6] * trail


def edge_fixtures(seed=2026):
    """Three chromosomes whose regions sit at their ends.  Returns dict(names, seqs, reads: one list per chromosome sorted by start,
    regions: (chromosome, start, stop) in pool order).  In pool order the region at the end of chrA is followed by the region at the
    start of chrB.  Every event's position is chosen so that a path that exists only at an edge is taken:
      chrA start  reads from position 0 (some with low-quality leading bases, some soft-clipped in front of the chromosome),
                  an insertion 12 and a deletion 30 bases from the start
      chrA middle homopolymer, {A,C}-only and ACG-repeat flanks (rejects of equal / low-complexity k-mers)
      chrA end    a tandem-repeat expansion (AL fallback) 80 bases before the end and 5 extra bases in the 14-base homopolymer that
                  ends the chromosome (equal k-mers, then the qend branch); reads end exactly at the end
      chrB start  a homopolymer run at position 0 with 5 extra bases
      chrB middle contigs that start 2 bases before a homopolymer with 5 extra bases (equal k-mers on both tries); 26-base reads
                  with an insertion: a contig shorter than K
      chrB end    contigs that start 20 bases before the end: 8 matching bases, a 5-base insertion, 12 matching bases, then bases
                  past the end -- a reference window shorter than K
      chrC        120 bp, shorter than one read, reads soft-clipped at both ends"""
    rng = np.random.default_rng(seed)
    names, seqs, reads, regions = ["chrA", "chrB", "chrC"], [], [[], [], []], []
    RL = 150

    # ---- chrA: 2600 bp
    a = list(random_seq(rng, 2600))
    a[1100:1145] = "A" * 45                                         # homopolymer
    a[1300:1380] = random_seq(rng, 80, "AC")                        # only A and C: every k-mer has < 3 distinct bases
    a[1600:1660] = "ACG" * 20                                       # 3-base repeat
    a[2520:2560] = "ACGTT" * 8                                      # tandem repeat 80..40 bases before the end
    a[2586:2600] = "A" * 14                                         # homopolymer that ends the chromosome
    A = "".join(a)
    seqs.append(A)
    ref0 = haplotype(A)
    alt0 = haplotype(A, [(12, "I", "GTTCA"), (30, "D", 6)])
    clip0 = haplotype(A, [(12, "I", "GTTCA"), (30, "D", 6)], lead="TGCAT")
    for k, at in enumerate([0, 0, 0, 1, 2, 4, 6, 9]):
        reads[0].append(hap_read(alt0, at, RL, qual=_lowq(RL, lead=6 if k % 3 == 1 else 0)))
    for at in (0, 0, 3, 5, 8, 11):
        reads[0].append(hap_read(ref0, at, RL, qual=_lowq(RL, lead=5 if at == 3 else 0)))
    for k in range(4):
        reads[0].append(hap_read(clip0, 0, RL, mapq=60 if k else 35))
    regions.append((0, 0, 40))
    # middle: equal / low-complexity k-mers
    mid = haplotype(A, [(1110, "I", "AAAAA"), (1200, "D", 3), (1330, "D", 6), (1615, "I", "ACGACG")])
    for at in range(980, 1500, 12):
        reads[0].append(hap_read(mid if (at // 12) % 3 else ref0, at, RL))
    regions.append((0, 1100, 1380))
    for at in range(1500, 1640, 10):
        reads[0].append(hap_read(mid if (at // 10) % 3 else ref0, at, RL))
    regions.append((0, 1600, 1640))
    # end: a tandem-repeat expansion (AL fallback) and 5 extra bases in the 14-base homopolymer that ends the chromosome: both k-mers
    # equal at first, the second try reaches past the contig's end and takes the qend branch; every read ends at or before the end
    endA = haplotype(A, [(2520, "I", "ACGTT"), (2586, "I", "AAAAA")])
    for k, back in enumerate([150, 150, 150, 150, 153, 157, 160, 164, 168]):
        reads[0].append(hap_read(endA, len(endA) - back, RL, qual=_lowq(RL, trail=4 if k == 5 else 0)))
    for back in (150, 150, 152, 156, 161, 166):
        reads[0].append(hap_read(ref0, 2600 - back, RL))
    regions.append((0, 2520, 2600))

    # ---- chrB: 2000 bp, a homopolymer at position 0 and contigs starting 20 bases before the end
    b = list(random_seq(rng, 2000))
    b[0:45] = "A" * 45
    b[998:1040] = "GC" + "A" * 40                                   # contigs start 2 bases before a homopolymer: equal k-mers twice
    B = "".join(b)
    seqs.append(B)
    altB = haplotype(B, [(0, "I", "AAAAA")])
    refB = haplotype(B)
    for at in (0, 0, 0, 2, 4, 7):
        reads[1].append(hap_read(altB, at, RL))
    for at in (0, 0, 3, 6):
        reads[1].append(hap_read(refB, at, RL))
    regions.append((1, 0, 45))
    altB2 = haplotype(B, [(1000, "I", "AAAAA")])
    for _ in range(5):
        reads[1].append(hap_read(altB2, 998, RL))
    for at in (990, 994, 1001, 1004):
        reads[1].append(hap_read(refB, at, RL))
    regions.append((1, 995, 1045))
    short = haplotype(B, [(1510, "I", "TCA")])                    # 26-base reads: a contig shorter than K (it aligns under -c 26)
    for _ in range(6):
        reads[1].append(hap_read(short, 1500, 26))
    regions.append((1, 1505, 1515))
    tailB = random_seq(rng, 140)
    shortwin = haplotype(B, [(1988, "I", "CTTAG")], tail=tailB)
    at = len(shortwin) - len(tailB) - 25                       # 8 + 5 + 12 bases before the end
    for _ in range(6):
        reads[1].append(hap_read(shortwin, at, RL))
    refBe = haplotype(B, tail=tailB)
    for back in (150, 147, 143, 140):
        reads[1].append(hap_read(refBe, len(refBe) - len(tailB) - back, RL))
    regions.append((1, 1970, 2000))

    # ---- chrC: 120 bp, shorter than one read
    C_ = random_seq(rng, 120)
    seqs.append(C_)
    lead, trail = random_seq(rng, 20), random_seq(rng, 20)
    altC = haplotype(C_, [(60, "D", 6)], lead=lead, tail=trail)
    refC = haplotype(C_, lead=lead, tail=trail)
    for k in range(6):
        reads[2].append(hap_read(altC, k % 3, 150 - 6 - (k % 3) * 2))
    for k in range(4):
        reads[2].append(hap_read(refC, k % 2, 150 - (k % 2)))
    regions.append((2, 0, 120))
    for r in reads:
        r.sort(key=lambda x: x["start"])
    return dict(names=names, seqs=seqs, reads=reads, regions=regions)


def edge_rois(fx, extra=None):
    """the fixtures as one Rois: a region holds the reads of its chromosome that overlap it (src/indelope.nim:449-452).  extra: optional
    (name, sequence, arrays of a one-chromosome region set) appended as a fourth chromosome"""
    sets, chroms = [], []
    for c, lo, hi in fx["regions"]:
        rr = [r for r in fx["reads"][c] if not (r["start"] > hi) and not (r["stop"] < lo)]
        sets.append(rois_from_reads(rr, fx["seqs"][c], roi_start=lo, roi_stop=hi)[1]); chroms.append(c)
    names, seqs = list(fx["names"]), list(fx["seqs"])
    if extra is not None:
        sets.append(extra[2]); chroms.append(len(names)); names.append(extra[0]); seqs.append(extra[1])
    arrays = merge_rois(sets, chroms, names, seqs)
    return host.Rois(arrays=arrays), arrays


def edge_files(fx, directory):
    """the fixtures as <directory>/edges.fa and <directory>/edges.bam (records with S operations, BGZF)"""
    fa, bam = os.path.join(str(directory), "edges.fa"), os.path.join(str(directory), "edges.bam")
    with open(fa, "w") as f:
        for n, s in zip(fx["names"], fx["seqs"]):
            f.write(">%s\n%s\n" % (n, "\n".join(s[i:i + 60] for i in range(0, len(s), 60))))
    recs = [bam_record(c, r["start"], r["cigar"], r["seq"], qual=r["qual"], mapq=r["mapq"], flag=r["flag"], name=b"e%d_%d" % (c, k))
            for c, rr in enumerate(fx["reads"]) for k, r in enumerate(rr)]
    with open(bam, "wb") as f:
        f.write(bgzf_compress(bam_bytes([(n, len(s)) for n, s in zip(fx["names"], fx["seqs"])], recs)))
    return fa, bam


def out_dir():
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(d, exist_ok=True)
    return d


# ---------------------------------------------------------------------------------------------------------------
# BAM files made and parsed with struct + zlib alone (SAM spec 4.1, 4.2): the independent side of the idl_bam_* tests
# ---------------------------------------------------------------------------------------------------------------
import struct
import zlib

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
SEQ16 = "=ACMGRSVTWYHKDBN"
CIG_OPS = "MIDNSHP=X"


def bgzf_member(chunk, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    c = co.compress(chunk) + co.flush()
    bsize = 18 + len(c) + 8 - 1
    assert bsize < 65536
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize) + c + struct.pack("<II", zlib.crc32(chunk), len(chunk)))


def bgzf_compress(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, block=0xff00, levels=None, eof=True):
    """data -> BGZF; `levels` cycles (level, strategy) pairs over the members so that one file holds stored, fixed and dynamic blocks"""
    out, k = [], 0
    for at in range(0, len(data), block):
        lv, st = (levels[k % len(levels)] if levels else (level, strategy)); k += 1
        chunk = data[at:at + block]
        if lv == 0 and len(chunk) > 0xff00 - 64:
            lv = 1  # a stored member must still fit 64 KiB with its framing
        out.append(bgzf_member(chunk, lv, st))
    if eof:
        out.append(BGZF_EOF)
    return b"".join(out)


def bam_record(ref_id, pos, cigar, seq, qual=None, mapq=60, flag=0, name=b"r", next_ref=-1, next_pos=-1, tlen=0, tags=b""):
    """cigar: list of (op char, len); seq: str over SEQ16"""
    l_seq = len(seq)
    nib = [SEQ16.index(c) for c in seq]
    if l_seq & 1:
        nib.append(0)
    packed = bytes(nib[i] << 4 | nib[i + 1] for i in range(0, len(nib), 2))
    qual = bytes([30] * l_seq) if qual is None else bytes(qual)
    assert len(qual) == l_seq
    cg = b"".join(struct.pack("<I", ln << 4 | CIG_OPS.index(op)) for op, ln in cigar)
    nm = name + b"\0"
    body = struct.pack("<iiBBHHHiiii", ref_id, pos, len(nm), mapq, 0, len(cigar), flag, l_seq, next_ref, next_pos, tlen) + nm + cg + packed + qual + tags
    return struct.pack("<i", len(body)) + body


def bam_bytes(refs, records, text=None):
    """refs: list of (name, length); records: list of bytes from bam_record -> the uncompressed BAM stream"""
    text = ("@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % r for r in refs)).encode() if text is None else text
    out = [b"BAM\1", struct.pack("<i", len(text)), text, struct.pack("<i", len(refs))]
    for name, ln in refs:
        nm = name.encode() + b"\0"
        out.append(struct.pack("<i", len(nm)) + nm + struct.pack("<i", ln))
    return b"".join(out) + b"".join(records)


def parse_bam(data):
    """uncompressed BAM stream -> header + per-record arrays as idl_bam_fetch lays them out (records without a target dropped)"""
    assert data[:4] == b"BAM\1"
    l_text, = struct.unpack_from("<i", data, 4)
    text = data[8:8 + l_text].decode()
    at = 8 + l_text
    n_ref, = struct.unpack_from("<i", data, at); at += 4
    refs = []
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", data, at); at += 4
        name = data[at:at + l_name - 1].decode(); at += l_name
        ln, = struct.unpack_from("<i", data, at); at += 4
        refs.append((name, ln))
    cols = dict(chrom=[], start=[], stop=[], len=[], mapq=[], flag=[])
    seq_off, cig_off, bases, quals, cigar = [0], [0], [], [], []
    n_unplaced = 0
    while at < len(data):
        bs, ref_id, pos, l_name, mapq, _bin, n_cig, flag, l_seq = struct.unpack_from("<iiiBBHHHi", data, at)
        b = at + 4; at += 4 + bs
        if ref_id < 0:
            n_unplaced += 1
            continue
        cg = struct.unpack_from("<%dI" % n_cig, data, b + 32 + l_name)
        rlen = sum(c >> 4 for c in cg if (c & 15) in (0, 2, 3, 7, 8))
        if (flag & 4) or n_cig == 0 or rlen == 0:
            rlen = 1
        so = b + 32 + l_name + 4 * n_cig
        packed = np.frombuffer(data, dtype=np.uint8, count=(l_seq + 1) // 2, offset=so)
        nib = np.empty(2 * len(packed), dtype=np.uint8); nib[0::2] = packed >> 4; nib[1::2] = packed & 15
        bases.append(np.frombuffer(SEQ16.encode(), dtype=np.uint8)[nib[:l_seq]])
        quals.append(np.frombuffer(data, dtype=np.uint8, count=l_seq, offset=so + (l_seq + 1) // 2))
        cigar.extend(cg)
        for k, v in zip(("chrom", "start", "stop", "len", "mapq", "flag"), (ref_id, pos, pos + rlen, l_seq, mapq, flag)):
            cols[k].append(v)
        seq_off.append(seq_off[-1] + l_seq); cig_off.append(cig_off[-1] + n_cig)
    out = dict(chrom=np.array(cols["chrom"], np.int32), start=np.array(cols["start"], np.int32), stop=np.array(cols["stop"], np.int32), len=np.array(cols["len"], np.int32),
               mapq=np.array(cols["mapq"], np.uint8), flag=np.array(cols["flag"], np.uint16), seq_off=np.array(seq_off, np.int64), cig_off=np.array(cig_off, np.uint64),
               bases=np.concatenate(bases) if bases else np.zeros(0, np.uint8), quals=np.concatenate(quals) if quals else np.zeros(0, np.uint8),
               cigar=np.array(cigar, np.uint32))
    return text, refs, out, n_unplaced


# ---------------------------------------------------------------------------------------------------------------
# Capacity limits: the oracle's per-region L lines (dump bit 64), region subsets, and directed regions built to sit exactly on a limit
# ---------------------------------------------------------------------------------------------------------------
DUMP_LIMITS = 64  # oracle only: "L <region> max_len=<longest contig of assemble + combine> max_corr=<most voting sites of one merge>"


def limits(odump):
    """{region ordinal: (longest contig, most voting sites)} from an oracle dump made with DUMP_LIMITS"""
    out = {}
    for l in odump.splitlines():
        if l.startswith("L\t"):
            f = l.split("\t")
            out[int(f[1])] = (int(f[2].split("=")[1]), int(f[3].split("=")[1]))
    return out


def by_region(dump, types="RCAE"):
    """{region ordinal: [lines]} of the per-region record types"""
    out = {}
    for l in dump.splitlines():
        if l[:1] in types:
            out.setdefault(int(l.split("\t")[1]), []).append(l)
    return out


def region_subset(arrays, keep):
    """the same reads and chromosomes with only the regions whose index is in `keep` (in order)"""
    keep = np.asarray(sorted(keep), np.int64)
    out = dict(arrays)
    for k in ("roi_chrom", "roi_start", "roi_stop", "roi_read_begin", "roi_n_reads"):
        out[k] = np.asarray(arrays[k])[keep]
    return out


def redraw_mapq(arrays, seed=7):
    """every read's MAPQ drawn again over 0-255, weighted toward the gates of the calling path (5/6, 9/10, 19/20) and toward 255"""
    rng = np.random.default_rng(seed)
    n = len(arrays["mapq"])
    edges = np.array([5, 6, 9, 10, 19, 20, 255], np.uint8)
    pick = rng.random(n)
    m = rng.integers(0, 256, n).astype(np.uint8)
    m = np.where(pick < 0.45, edges[rng.integers(0, len(edges), n)], m)
    m = np.where((pick >= 0.45) & (pick < 0.6), np.uint8(255), m)
    out = dict(arrays)
    out["mapq"] = m
    return out


def tiled_region(ref, at, span, read_len, step, hap=None, mapq=60, last_len=None):
    """reads of `read_len` bases every `step` bases from `at` (of `hap`, the reference by default), the last one `last_len` long, so that
    they assemble into one contig of exactly `span` bases: each read overlaps the contig by read_len - step >= 0.88 of its length"""
    src = ref if hap is None else hap
    reads, s = [], at
    while True:
        n = at + span - s
        if n <= (last_len or read_len) + step - 1:           # the last read: read_len .. read_len + step - 1 bases
            reads.append(dict(start=s, seq=src[s:s + n], mapq=mapq))
            break
        reads.append(dict(start=s, seq=src[s:s + read_len], mapq=mapq))
        s += step
    assert reads[-1]["start"] + len(reads[-1]["seq"]) == at + span
    return reads


def cap_fixture(cap, seed=11):
    """regions around max_contig_len = cap, in pool order: [0] reads tiling exactly cap bases (called), [1] exactly cap + 1 bases (the merge
    check drops it), and when cap + 1 fits max_read_len, [2] five copies of one read of cap bases (called) and [3] of cap + 1 bases (the
    read-trim check drops it); a region with a 12-base deletion at the end keeps the batch calling a variant"""
    rng = np.random.default_rng(seed)
    ref = random_seq(rng, 3 * cap + 12000)
    sets, at = [], 1000
    for span in (cap, cap + 1):
        reads = tiled_region(ref, at, span, 100, 10)
        sets.append(rois_from_reads(reads, ref, roi_start=at + 40, roi_stop=at + 60)[1]); at += span + 1000
    if cap < 512:
        for n in (cap, cap + 1):
            reads = [dict(start=at, seq=ref[at:at + n]) for _ in range(5)]
            sets.append(rois_from_reads(reads, ref, roi_start=at + 40, roi_stop=at + 60)[1]); at += n + 1000
    hap = ref[:at + 100] + ref[at + 112:]
    reads = [dict(start=at + i, seq=(hap if (i // 3) % 2 else ref)[at + i:at + i + 100]) for i in range(30, 72, 3)]
    sets.append(rois_from_reads(reads, ref, roi_start=at + 90, roi_stop=at + 120)[1])
    return merge_rois(sets)


def length_fixture(lengths, seed=3, mapqs=None):
    """one region per entry of `lengths` (a list of read lengths): reads of those lengths, alternately from the reference and from a haplotype
    with a 12-base deletion in a tandem repeat, all overlapping the deletion; qualities 30, so every trimmed length equals the read's length.  mapqs: optional
    per-region list of MAPQs (cycled over the reads)"""
    rng = np.random.default_rng(seed)
    sets, ref_parts, off = [], [], 0
    for k, lens in enumerate(lengths):
        L = max(lens)
        seg = random_seq(rng, 2 * L + 400)
        d = L + 200                                   # deletion of seg[d:d + 12]: two units of a 6-base tandem repeat (the AL fallback)
        seg = seg[:d - 24] + "ACGTTG" * 10 + seg[d + 36:]
        hap = seg[:d] + seg[d + 12:]
        reads = []
        for i, n in enumerate(lens):
            lo, hi = max(0, d - n + 20), d - 20       # the read covers the deletion with >= 20 bases on each side
            s = lo + (i * 7919) % max(1, hi - lo)
            src = hap if i % 2 else seg
            r = dict(start=off + s, seq=src[s:s + n])
            if mapqs is not None:
                r["mapq"] = int(mapqs[k][i % len(mapqs[k])])
            reads.append(r)
        reads.sort(key=lambda r: r["start"])
        ref_parts.append(seg)
        sets.append((reads, off + d - 10, off + d + 22))
        off += len(seg)
    ref = "".join(ref_parts)
    return merge_rois([rois_from_reads(r, ref, roi_start=a, roi_stop=b)[1] for r, a, b in sets])


def corr_fixture(sites=(128, 129), seed=13):
    """one region per entry of `sites`: a 500-base read with three 100-base copies of its start (a contig of 4 reads whose last 400 bases
    have support 1) and four copies of a 499-base read one base to the right that differs from it at `n` positions of those 400 bases.
    The two contigs stay apart in assemble (a single read never votes) and merge in the first combine pass with exactly n voting sites,
    every one allowed (support 4 against 1, both contigs of 4 reads)"""
    rng = np.random.default_rng(seed)
    sets, parts, off = [], [], 0
    for n in sites:
        seg = random_seq(rng, 1000)
        a = seg[200:700]
        b = list(seg[201:700])
        for k in range(n):
            p = 120 + 2 * k - 1                              # position 120 + 2k of the long read
            b[p] = "ACGT"[("ACGT".index(b[p]) + 1 + k % 3) % 4]
        b = "".join(b)
        reads = [dict(start=off + 200, seq=a)] + [dict(start=off + 200, seq=a[:100]) for _ in range(3)] + \
                [dict(start=off + 201, seq=b) for _ in range(4)]
        sets.append((reads, off + 400, off + 420))
        parts.append(seg); off += len(seg)
    ref = "".join(parts)
    return merge_rois([rois_from_reads(r, ref, roi_start=lo, roi_stop=hi)[1] for r, lo, hi in sets])


def long_contig_fixture(spans=(6000, 4900), seed=17):
    """one region per entry of `spans`: 250-base reads every 20 bases of a haplotype with a 12-base deletion in the middle, which assemble
    into one contig of about `span` bases aligned to a window about as long (call-site A, band 50)"""
    rng = np.random.default_rng(seed)
    sets, parts, off = [], [], 0
    for span in spans:
        seg = random_seq(rng, span + 1000)
        d = 500 + span // 2
        hap = seg[:d] + seg[d + 12:]
        reads = tiled_region(hap, 500, span, 250, 20)
        for r in reads:
            r["start"] += off
            if r["start"] - off + len(r["seq"]) > d:
                r["stop"] = r["start"] + len(r["seq"]) + (12 if r["start"] - off < d else 0)
        sets.append((reads, off + d - 10, off + d + 22))
        parts.append(seg); off += len(seg)
    ref = "".join(parts)
    return merge_rois([rois_from_reads(r, ref, roi_start=lo, roi_stop=hi)[1] for r, lo, hi in sets])
