"""ctypes binding of libindelope_host.so (include/indelope_host.h): synthetic data, the gen_roi sweep
(src/indelope.nim:430-545), batch packing and the VCF cascade (src/indelope.nim:375-428)."""
import ctypes as C
import os

import numpy as np

from . import build as _build
from .abi import Batch, Params, Results, default_params  # noqa: F401

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)


class RoiSetC(C.Structure):
    _fields_ = [
        ("n_reads", C.c_int64), ("start", i32p), ("stop", i32p), ("mapq", u8p), ("flag", u16p), ("len", i32p),
        ("seq_off", i64p), ("bases", u8p), ("quals", u8p),
        ("n_rois", C.c_int64), ("roi_chrom", i32p), ("roi_start", i32p), ("roi_stop", i32p), ("roi_read_begin", i64p),
        ("roi_n_reads", i32p), ("read_idx", i64p),
        ("n_chroms", C.c_int32), ("chrom_name", C.POINTER(C.c_char_p)), ("chrom_seq", C.POINTER(u8p)), ("chrom_len", i64p),
    ]


class ChromReads(C.Structure):
    _fields_ = [("first_read", C.c_int64), ("n_reads", C.c_int64), ("chrom_len", C.c_int32), ("start", i32p), ("stop", i32p), ("flag", u16p),
                ("cigar", u32p), ("cig_off", C.POINTER(C.c_uint64))]


class SynthParams(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("n_chroms", C.c_int32), ("chrom_len", C.c_int64), ("n_events", C.c_int32), ("min_indel", C.c_int32),
        ("max_indel", C.c_int32), ("coverage", C.c_double), ("read_len", C.c_int32), ("sub_rate", C.c_double), ("tr_fraction", C.c_double),
        ("tr_max_unit", C.c_int32), ("het_fraction", C.c_double), ("lowq_tail_fraction", C.c_double), ("low_mapq_fraction", C.c_double),
        ("dup_fraction", C.c_double), ("n_base_rate", C.c_double), ("locus_only", C.c_int32), ("locus_flank", C.c_int32),
        ("max_cigar_indel", C.c_int32), ("min_cigar_flank", C.c_int32), ("chrom_first", C.c_int32), ("qual_levels", C.c_int32),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = _build.build_host()
        L = C.CDLL(path)
        L.idlh_synth.restype = C.c_void_p
        L.idlh_synth.argtypes = [C.POINTER(SynthParams)]
        L.idlh_dataset_free.argtypes = [C.c_void_p]
        L.idlh_dataset_counts.argtypes = [C.c_void_p, i64p]
        L.idlh_dataset_truth.argtypes = [C.c_void_p, i64p, C.c_int64]
        L.idlh_dataset_truth.restype = C.c_int64
        L.idlh_load.restype = C.c_void_p
        L.idlh_load.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]
        L.idlh_load_region.restype = C.c_void_p
        L.idlh_load_fasta.restype = C.c_void_p
        L.idlh_load_fasta.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
        L.idlh_dataset_set_targets.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_char_p), i64p, C.c_char_p, C.c_size_t]
        L.idlh_dataset_set_bam_targets.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_size_t]
        L.idlh_dataset_from_sequences.restype = C.c_void_p
        L.idlh_dataset_from_sequences.argtypes = [C.c_int32, C.POINTER(C.c_char_p), C.POINTER(u8p), i64p]
        L.idlh_load_region.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_char_p, C.c_size_t]
        L.idlh_write_fasta.argtypes = [C.c_void_p, C.c_char_p]
        L.idlh_write_bam.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.idlh_stream_open.restype = C.c_void_p
        L.idlh_stream_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_size_t]
        L.idlh_stream_next.restype = C.c_void_p
        L.idlh_stream_next.argtypes = [C.c_void_p, C.c_int64, C.c_char_p, C.c_size_t]
        L.idlh_stream_targets.restype = C.c_void_p
        L.idlh_stream_targets.argtypes = [C.c_void_p]
        L.idlh_stream_counts.argtypes = [C.c_void_p, i64p]
        L.idlh_stream_close.argtypes = [C.c_void_p]
        L.idlh_dataset_chrom.restype = C.POINTER(ChromReads)
        L.idlh_dataset_chrom.argtypes = [C.c_void_p, C.c_int32]
        L.idlh_chrom_free.argtypes = [C.POINTER(ChromReads)]
        L.idlh_sweep.restype = C.c_void_p
        L.idlh_sweep.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
        L.idlh_rois_free.argtypes = [C.c_void_p]
        L.idlh_rois_view.restype = C.POINTER(RoiSetC)
        L.idlh_rois_view.argtypes = [C.c_void_p]
        L.idlh_pack_size.argtypes = [C.POINTER(RoiSetC), C.c_int64, C.c_int64, C.POINTER(Params), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.idlh_pack.argtypes = [C.POINTER(RoiSetC), C.c_int64, C.c_int64, C.POINTER(Params), C.POINTER(Batch)]
        L.idlh_batch_alloc_host.restype = C.POINTER(Batch)
        L.idlh_batch_alloc_host.argtypes = [C.c_size_t] * 4
        L.idlh_batch_free_host.argtypes = [C.POINTER(Batch)]
        L.idlh_unpack.argtypes = [u32p, u32p, C.c_uint64, C.c_int32, C.c_char_p]
        L.idlh_vcf_new.restype = C.c_void_p
        L.idlh_vcf_free.argtypes = [C.c_void_p]
        L.idlh_vcf_header.restype = C.c_void_p
        L.idlh_vcf_header.argtypes = [C.POINTER(RoiSetC)]
        L.idlh_vcf_records.restype = C.c_void_p
        L.idlh_vcf_records.argtypes = [C.c_void_p, C.POINTER(RoiSetC), C.c_int64, C.POINTER(Params), C.POINTER(Results), C.c_int32, C.POINTER(C.c_void_p)]
        L.idlh_free.argtypes = [C.c_void_p]
        L.idlh_vcf_set_dedup.argtypes = [C.c_void_p, C.c_int]
        L.idlh_vcf_dedup.restype = C.c_void_p
        L.idlh_vcf_dedup.argtypes = [C.c_char_p]
        L.idlh_vcf_dedup_inplace.restype = C.c_size_t
        L.idlh_vcf_dedup_inplace.argtypes = [C.c_void_p, C.c_size_t]
        L.idlh_vcf_dedup_n.restype = C.c_void_p
        L.idlh_vcf_dedup_n.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.idlh_set_threads.argtypes = [C.c_int]
        L.idlh_vcf_status_counts.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.idlh_trim.argtypes = [u8p, C.c_int32, i32p]
        L.idlh_trim.restype = C.c_int32
        _lib = L
    return _lib


def _take(ptr):
    s = C.string_at(ptr).decode()
    lib().idlh_free(ptr)
    return s


def synth_params(**kw):
    p = SynthParams()
    lib().idlh_default_synth(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


# The five BASELINE.json configs as generator settings (SURVEY.md 8d).  `locus_only` simulates reads only around
# planted events (locus_flank bases either side, > read length + the longest CIGAR indel, so every read that can
# overlap a region of interest exists): reads elsewhere carry no CIGAR event, never enter a region of interest and so
# never reach the path this repo implements.  Event counts can be scaled down for tests.
CONFIGS = {
    # 1 Mb, 30x, 200 planted 5-300 bp indels, whole contig simulated (the reference's CPU-runnable case)
    "pr1": dict(seed=20171101, n_chroms=1, chrom_len=1_000_000, n_events=200, coverage=30.0, read_len=150, locus_only=0),
    # exome: ~2000 indels inside targets at 100x (2x150 pairs act as independent reads on this path)
    "exome": dict(seed=20171102, n_chroms=1, chrom_len=50_000_000, n_events=2000, coverage=100.0, read_len=150, locus_only=1, locus_flank=220),
    # chr1-sized 30x WGS: 1 indel per 5 kb + 1 tandem-repeat event per 20 kb
    "chr1": dict(seed=20171103, n_chroms=1, chrom_len=248_000_000, n_events=62_000, coverage=30.0, read_len=150, locus_only=1, locus_flank=220, tr_fraction=0.2),
    # 500x panel rich in tandem repeats / homopolymers
    "panel500": dict(seed=20171104, n_chroms=1, chrom_len=2_000_000, n_events=400, coverage=500.0, read_len=150, locus_only=1, locus_flank=220, tr_fraction=0.6,
                     tr_max_unit=3, max_indel=60),
    # the same panel at a lower substitution rate (2e-4 per base): most deep regions then stay at or under the 20-contig gate of
    # src/indelope.nim:209, so regions of hundreds of reads reach the contig alignment, the k-mer pass and -- tandem repeats --
    # the AL fallback with hundreds of reads per event (config 4's "survivors", SURVEY.md 8d.4)
    "panel500_lowerr": dict(seed=20171104, n_chroms=1, chrom_len=2_000_000, n_events=400, coverage=500.0, read_len=150, locus_only=1, locus_flank=220,
                            tr_fraction=0.6, tr_max_unit=3, max_indel=60, sub_rate=2e-4),
    # 30x whole genome, 3.1 Gb over 24 contigs: one rank's interval shard is built with n_chroms/chrom_len per shard
    "wgs": dict(seed=20171105, n_chroms=1, chrom_len=129_000_000, n_events=32_000, coverage=30.0, read_len=150, locus_only=1, locus_flank=220,
                tr_fraction=0.2),
}


class Dataset:
    """synthetic reference + coordinate-sorted reads (the BAM/FASTA stand-in)"""

    def __init__(self, params=None, _handle=None, **kw):
        if _handle is not None:
            self.params, self.h = None, _handle
        else:
            self.params = params if params is not None else synth_params(**kw)
            self.h = lib().idlh_synth(C.byref(self.params))
        c = (C.c_int64 * 4)()
        lib().idlh_dataset_counts(self.h, c)
        self.n_reads, self.n_bases, self.n_events, self.n_chroms = list(c)

    @classmethod
    def load(cls, fasta, bam, threads=1):
        """reference FASTA + coordinate-sorted BAM from disk (libindelope_host's own BGZF/BAM reader)"""
        err = C.create_string_buffer(512)
        h = lib().idlh_load(str(fasta).encode(), str(bam).encode(), threads, err, 512)
        if not h:
            raise IOError(err.value.decode())
        return cls(_handle=h)

    @classmethod
    def load_region(cls, fasta, bam, target, beg=0, end=0):
        """`b.querys("target:beg-end")` through <bam>.bai: only the records overlapping [beg, end) of `target` (0-based, half open)"""
        err = C.create_string_buffer(512)
        h = lib().idlh_load_region(str(fasta).encode(), str(bam).encode(), str(target).encode(), beg, end, err, 512)
        if not h:
            raise IOError(err.value.decode())
        return cls(_handle=h)

    @classmethod
    def load_fasta(cls, fasta):
        """the reference sequences alone (the BAM is decoded on the device: cuda.Bam); the FASTA plain or compressed with bgzip"""
        err = C.create_string_buffer(512)
        h = lib().idlh_load_fasta(str(fasta).encode(), err, 512)
        if not h:
            raise IOError(err.value.decode())
        return cls(_handle=h)

    @classmethod
    def from_sequences(cls, names, seqs):
        """a reference without reads from names and sequences (bytes / uint8 arrays), e.g. those of a cuda.Fasta; everything is copied"""
        a = [np.ascontiguousarray(np.frombuffer(x, np.uint8) if isinstance(x, (bytes, bytearray)) else x, dtype=np.uint8) for x in seqs]
        n = len(a)
        nm = (C.c_char_p * max(n, 1))(*[x.encode("latin-1") for x in names])
        sp = (u8p * max(n, 1))(*[x.ctypes.data_as(u8p) for x in a])
        lens = np.array([len(x) for x in a] or [0], dtype=np.int64)
        return cls(_handle=lib().idlh_dataset_from_sequences(n, nm, sp, lens.ctypes.data_as(i64p)))

    def set_bam_targets(self, bam):
        """set_targets with the targets of a BAM file's header (only the header's members are read)"""
        err = C.create_string_buffer(512)
        if lib().idlh_dataset_set_bam_targets(self.h, str(bam).encode(), err, 512) != 0:
            raise IOError(err.value.decode())
        c = (C.c_int64 * 4)()
        lib().idlh_dataset_counts(self.h, c)
        self.n_reads, self.n_bases, self.n_events, self.n_chroms = list(c)

    def set_targets(self, names, lengths):
        """order the sequences as a BAM header lists its targets (same checks and messages as Dataset.load)"""
        n = len(names)
        arr = (C.c_char_p * n)(*[s.encode() for s in names])
        lens = np.ascontiguousarray(lengths, dtype=np.int64)
        err = C.create_string_buffer(512)
        if lib().idlh_dataset_set_targets(self.h, n, arr, lens.ctypes.data_as(i64p), err, 512) != 0:
            raise IOError(err.value.decode())
        c = (C.c_int64 * 4)()
        lib().idlh_dataset_counts(self.h, c)
        self.n_reads, self.n_bases, self.n_events, self.n_chroms = list(c)

    def sequences(self):
        """(names, sequences as uint8 arrays): views of the dataset's memory -- keep the dataset alive"""
        r = Rois(lib().idlh_sweep(self.h, 255, 1 << 30, 1 << 30), self)   # no regions: just the views
        a = r.arrays()
        self._seq_owner = r
        return a["chrom_names"], a["chrom_seqs"]

    def write_fasta(self, path):
        """FASTA (60 columns) + path.fai"""
        if lib().idlh_write_fasta(self.h, str(path).encode()) != 0:
            raise IOError("cannot write %s" % path)

    def write_bam(self, path, level=1):
        """coordinate-sorted BAM of the reads (BGZF, deflate level 0-9)"""
        if lib().idlh_write_bam(self.h, str(path).encode(), level) != 0:
            raise IOError("cannot write %s" % path)

    def chrom_reads(self, chrom):
        """records of one chromosome as numpy arrays (copies): first_read, chrom_len, start, stop, flag, cigar, cig_off -- the input of cuda.sweep"""
        p = lib().idlh_dataset_chrom(self.h, chrom)
        if not p:
            raise IndexError(chrom)
        c = p.contents
        n = int(c.n_reads)
        def arr(ptr, m, t):
            return np.ctypeslib.as_array(ptr, shape=(m,)).astype(t, copy=True) if m else np.zeros(0, t)
        off = arr(c.cig_off, n + 1, np.uint64)
        out = dict(first_read=int(c.first_read), chrom_len=int(c.chrom_len), start=arr(c.start, n, np.int32), stop=arr(c.stop, n, np.int32),
                   flag=arr(c.flag, n, np.uint16), cig_off=off, cigar=arr(c.cigar, int(off[-1]) if n else 0, np.uint32))
        lib().idlh_chrom_free(p)
        return out

    def truth(self):
        out = np.zeros((max(self.n_events, 1), 6), dtype=np.int64)
        lib().idlh_dataset_truth(self.h, out.ctypes.data_as(i64p), self.n_events)
        return out[:self.n_events]

    def sweep(self, min_reads=3, max_read_coverage=600):
        """gen_roi for every target with the CLI's settings (src/indelope.nim:602): min_event_support = max(3, min_reads-2)"""
        return Rois(lib().idlh_sweep(self.h, max(3, min_reads - 2), min_reads, max_read_coverage), self)

    def __del__(self):
        if getattr(self, "h", None):
            lib().idlh_dataset_free(self.h)
            self.h = None


class Stream:
    """FASTA + coordinate-sorted BAM swept front to back in bounded memory: groups of regions of interest, the same
    regions the whole-file sweep finds (idlh_stream_* in include/indelope_host.h)"""

    def __init__(self, fasta, bam, threads=1, min_reads=3, max_read_coverage=600):
        err = C.create_string_buffer(512)
        self.h = lib().idlh_stream_open(str(fasta).encode(), str(bam).encode(), threads, max(3, min_reads - 2), min_reads, max_read_coverage, err, 512)
        if not self.h:
            raise IOError(err.value.decode())

    def targets(self):
        return Rois(lib().idlh_stream_targets(self.h), self)

    def __iter__(self):
        return self.groups()

    def groups(self, target_reads=400000):
        while True:
            err = C.create_string_buffer(512)
            h = lib().idlh_stream_next(self.h, target_reads, err, 512)
            if not h:
                if err.value:
                    raise IOError(err.value.decode())
                return
            yield Rois(h, self)

    def counts(self):
        c = (C.c_int64 * 2)()
        lib().idlh_stream_counts(self.h, c)
        return int(c[0]), int(c[1])

    def __del__(self):
        if getattr(self, "h", None):
            lib().idlh_stream_close(self.h)
            self.h = None


def _arr(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).view(dtype)


class Rois:
    """regions of interest + their reads (flat arrays; zero-copy views of the C++ side)"""

    def __init__(self, handle=None, owner=None, arrays=None):
        self.h = handle
        self.owner = owner
        if handle is not None:
            self.c = lib().idlh_rois_view(handle).contents
        else:
            self._from_arrays(arrays)
        self.n_rois = int(self.c.n_rois)

    def _from_arrays(self, d):
        dt = dict(start=np.int32, stop=np.int32, mapq=np.uint8, flag=np.uint16, len=np.int32, seq_off=np.int64, bases=np.uint8, quals=np.uint8,
                  roi_chrom=np.int32, roi_start=np.int32, roi_stop=np.int32, roi_read_begin=np.int64, roi_n_reads=np.int32, read_idx=np.int64)
        self.d = {k: np.ascontiguousarray(d[k], dtype=t) for k, t in dt.items()}
        self.d["chrom_names"] = list(d["chrom_names"])
        self.d["chrom_seqs"] = [np.ascontiguousarray(s, dtype=np.uint8) for s in d["chrom_seqs"]]
        g = self.d
        r = RoiSetC()
        r.n_reads = len(g["start"])
        for k in ("start", "stop", "len", "roi_chrom", "roi_start", "roi_stop", "roi_n_reads"):
            setattr(r, k, g[k].ctypes.data_as(i32p))
        for k in ("seq_off", "roi_read_begin", "read_idx"):
            setattr(r, k, g[k].ctypes.data_as(i64p))
        r.mapq = g["mapq"].ctypes.data_as(u8p)
        r.flag = g["flag"].ctypes.data_as(u16p)
        r.bases = g["bases"].ctypes.data_as(u8p)
        r.quals = g["quals"].ctypes.data_as(u8p)
        r.n_rois = len(g["roi_start"])
        n = len(g["chrom_names"])
        self._names = (C.c_char_p * n)(*[s.encode() for s in g["chrom_names"]])
        self._seqs = (u8p * n)(*[s.ctypes.data_as(u8p) for s in g["chrom_seqs"]])
        self._lens = np.array([len(s) for s in g["chrom_seqs"]], dtype=np.int64)
        r.n_chroms = n
        r.chrom_name = self._names
        r.chrom_seq = self._seqs
        r.chrom_len = self._lens.ctypes.data_as(i64p)
        self.c = r

    def arrays(self):
        """dict of numpy views in the layout oracle.pyoracle.RoiSetArrays and Rois(arrays=...) take"""
        c = self.c
        n, m = int(c.n_reads), int(c.n_rois)
        nidx = int(np.sum(_arr(c.roi_n_reads, m, np.int32))) if m else 0
        nb = int(_arr(c.seq_off, n, np.int64)[-1] + _arr(c.len, n, np.int32)[-1]) if n else 0
        lens = _arr(c.chrom_len, c.n_chroms, np.int64)
        return dict(
            start=_arr(c.start, n, np.int32), stop=_arr(c.stop, n, np.int32), mapq=_arr(c.mapq, n, np.uint8), flag=_arr(c.flag, n, np.uint16),
            len=_arr(c.len, n, np.int32), seq_off=_arr(c.seq_off, n, np.int64), bases=_arr(c.bases, nb, np.uint8), quals=_arr(c.quals, nb, np.uint8),
            roi_chrom=_arr(c.roi_chrom, m, np.int32), roi_start=_arr(c.roi_start, m, np.int32), roi_stop=_arr(c.roi_stop, m, np.int32),
            roi_read_begin=_arr(c.roi_read_begin, m, np.int64), roi_n_reads=_arr(c.roi_n_reads, m, np.int32), read_idx=_arr(c.read_idx, nidx, np.int64),
            chrom_names=[c.chrom_name[i].decode() for i in range(c.n_chroms)],
            chrom_seqs=[_arr(c.chrom_seq[i], int(lens[i]), np.uint8) for i in range(c.n_chroms)],
        )

    def total_reads(self, lo=0, hi=None):
        hi = self.n_rois if hi is None else hi
        return int(np.sum(_arr(self.c.roi_n_reads, self.n_rois, np.int32)[lo:hi])) if self.n_rois else 0

    def pack_size(self, lo, hi, params):
        a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
        lib().idlh_pack_size(C.byref(self.c), lo, hi, C.byref(params), C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def pack(self, lo, hi, params, batch):
        """fill an idl_batch (from Context.batch_alloc or host_batch) with regions [lo, hi)"""
        rc = lib().idlh_pack(C.byref(self.c), lo, hi, C.byref(params), batch)
        if rc != 0:
            raise RuntimeError("idlh_pack failed: %d" % rc)

    def header(self):
        return _take(lib().idlh_vcf_header(C.byref(self.c)))

    def __del__(self):
        if getattr(self, "h", None):
            lib().idlh_rois_free(self.h)
            self.h = None


def bai_target_span(bam, target):
    """where one target's records lie in the file, from <bam>.bai: dict(file_begin, file_end, first_record, end_member, end_offset) or None when the index
    lists no record for the target -- the arguments of cuda.Bam(bytes[file_begin:file_end], slice=...)"""
    L = lib()
    v = [C.c_uint64() for _ in range(5)]
    err = C.create_string_buffer(512)
    L.idlh_bai_target_span.argtypes = [C.c_char_p, C.c_int32] + [C.POINTER(C.c_uint64)] * 5 + [C.c_char_p, C.c_size_t]
    rc = L.idlh_bai_target_span(str(bam).encode(), target, *[C.byref(x) for x in v], err, 512)
    if rc < 0:
        raise IOError(err.value.decode())
    if rc == 1:
        return None
    return dict(zip(("file_begin", "file_end", "first_record", "end_member", "end_offset"), (int(x.value) for x in v)))


def bai_region_run(bam, target, w0, w1):
    """idlh_bai_region_run: the records of `target` from the first record of 16 kb window w0 to the first record of window w1 + 1 (or to the target's end):
    dict(file_begin, file_end, first_record, end_member, end_offset, zone_lo, to_end) with empty=True when the run holds no record"""
    L = lib()
    v = [C.c_uint64() for _ in range(5)]
    zl, te = C.c_int64(), C.c_int32()
    err = C.create_string_buffer(512)
    L.idlh_bai_region_run.argtypes = [C.c_char_p, C.c_int32, C.c_int64, C.c_int64] + [C.POINTER(C.c_uint64)] * 5 + [C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.c_char_p, C.c_size_t]
    rc = L.idlh_bai_region_run(str(bam).encode(), target, w0, w1, *[C.byref(x) for x in v], C.byref(zl), C.byref(te), err, 512)
    if rc < 0:
        raise IOError(err.value.decode())
    out = dict(zip(("file_begin", "file_end", "first_record", "end_member", "end_offset"), (int(x.value) for x in v)))
    out.update(zone_lo=int(zl.value), to_end=bool(te.value), empty=rc == 1)
    return out


def parse_regions(ref_names, ref_len, regions=(), bed=None):
    """idlh_regions_parse: `-r` strings (chr[:beg[-end]], 1-based, inclusive) and a `-R` BED file (0-based, half open) -> one list of sorted, merged half-open
    (beg, end) intervals per target of the header.  ValueError with the reason for a malformed string, a bad BED line or a target not in the header."""
    L = lib()
    L.idlh_regions_parse.restype = C.c_void_p
    L.idlh_regions_parse.argtypes = [C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_int64), C.c_int32, C.POINTER(C.c_char_p), C.c_char_p, C.c_char_p, C.c_size_t]
    L.idlh_regions_get.restype = C.c_int64
    L.idlh_regions_get.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int64]
    L.idlh_regions_free.argtypes = [C.c_void_p]
    n = len(ref_names)
    names = (C.c_char_p * max(n, 1))(*[x.encode() for x in ref_names])
    lens = (C.c_int64 * max(n, 1))(*[int(x) for x in ref_len])
    regions = list(regions or [])
    rv = (C.c_char_p * max(len(regions), 1))(*[str(x).encode() for x in regions])
    err = C.create_string_buffer(512)
    h = L.idlh_regions_parse(n, names, lens, len(regions), rv, str(bed).encode() if bed else None, err, 512)
    if not h:
        raise ValueError(err.value.decode())
    try:
        out = []
        for c in range(n):
            k = L.idlh_regions_get(h, c, None, None, 0)
            b, e = (C.c_int64 * max(k, 1))(), (C.c_int64 * max(k, 1))()
            L.idlh_regions_get(h, c, b, e, k)
            out.append([(int(b[i]), int(e[i])) for i in range(k)])
        return out
    finally:
        L.idlh_regions_free(h)


def set_threads(n):
    """host threads of idlh_pack / idlh_pack_size (0 = $IDLH_THREADS, else every core up to 32)"""
    lib().idlh_set_threads(int(n))


def host_batch(max_regions, max_reads, max_seq_bases, max_ref_bases):
    return lib().idlh_batch_alloc_host(max_regions, max_reads, max_seq_bases, max_ref_bases)


def host_batch_free(b):
    lib().idlh_batch_free_host(b)


def unpack(pool2, pooln, off, n):
    buf = C.create_string_buffer(n + 1)
    lib().idlh_unpack(pool2, pooln, off, n, buf)
    return buf.value.decode()


def trim(quals):
    qa = np.ascontiguousarray(quals, dtype=np.uint8)
    n = C.c_int32()
    a = lib().idlh_trim(qa.ctypes.data_as(u8p), len(qa), C.byref(n))
    return a, n.value


class VcfWriter:
    """filter cascade + VCF text over device results, carrying the dedup state of src/indelope.nim:598-608 across batches"""

    def __init__(self, dedup=True):
        self.h = lib().idlh_vcf_new()
        lib().idlh_vcf_set_dedup(self.h, 1 if dedup else 0)

    def status_counts(self):
        """regions seen so far per idl_region_result.status bit (IDL_RS_*: index = bit number)"""
        out = (C.c_uint64 * 8)()
        lib().idlh_vcf_status_counts(self.h, out)
        return list(out)

    def records(self, rois, lo, params, results, dump_level=0):
        dump = C.c_void_p()
        p = lib().idlh_vcf_records(self.h, C.byref(rois.c), lo, C.byref(params), results, dump_level, C.byref(dump))
        return _take(p), _take(dump.value)

    def records_bytes(self, rois, lo, params, results):
        """the record text as bytes (no dump, no str round trip: a genome's records are tens of megabytes)"""
        p = lib().idlh_vcf_records(self.h, C.byref(rois.c), lo, C.byref(params), results, 0, None)
        out = C.string_at(p)
        lib().idlh_free(p)
        return out

    def __del__(self):
        if getattr(self, "h", None):
            lib().idlh_vcf_free(self.h)
            self.h = None


def dedup_inplace(ptr, n):
    """order-dependent dedup over n bytes at address ptr (n + 1 writable), in place; returns the new length"""
    return int(lib().idlh_vcf_dedup_inplace(ptr, n))


def dedup_records(text):
    """order-dependent dedup of src/indelope.nim:604-608 over merged record lines (str -> str, bytes-like -> bytes)"""
    if isinstance(text, str):
        return _take(lib().idlh_vcf_dedup(text.encode()))
    buf = (C.c_char * len(text)).from_buffer(text) if isinstance(text, bytearray) else C.create_string_buffer(bytes(text), len(text))
    n = C.c_size_t()
    p = lib().idlh_vcf_dedup_n(C.addressof(buf), len(text), C.byref(n))
    out = C.string_at(p, n.value)
    lib().idlh_free(p)
    return out
