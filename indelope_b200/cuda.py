"""ctypes binding of libindelope_cuda.so (include/indelope_cuda.h).  There is no CPU fallback: creating a
Context without a CUDA device raises, and so does a missing library."""
import ctypes as C
import os

import numpy as np

from . import build as _build
from .abi import (Batch, Ez, Params, Results, default_params)  # noqa: F401

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)

_lib = None


class IdlError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        path = _build.CUDA_LIB
        if not os.path.exists(path):
            path = _build.build_cuda()
        L = C.CDLL(path)
        L.idl_strerror.restype = C.c_char_p
        L.idl_last_cuda_error.restype = C.c_char_p
        L.idl_last_cuda_error.argtypes = [C.c_void_p]
        L.idl_create.argtypes = [C.c_int, C.POINTER(Params), C.POINTER(C.c_void_p)]
        L.idl_destroy.argtypes = [C.c_void_p]
        L.idl_batch_alloc.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.POINTER(Batch))]
        L.idl_batch_free.argtypes = [C.c_void_p, C.POINTER(Batch)]
        L.idl_submit.argtypes = [C.c_void_p, C.POINTER(Batch), u64p]
        L.idl_upload.argtypes = [C.c_void_p, C.POINTER(Batch)]
        L.idl_run_resident.argtypes = [C.c_void_p, C.POINTER(Batch), u64p]
        L.idl_wait.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.POINTER(Results))]
        L.idl_release.argtypes = [C.c_void_p, C.c_uint64]
        L.idl_default_params.argtypes = [C.POINTER(Params)]
        L.idl_ksw2_batch.argtypes = [C.c_void_p, C.c_size_t, u8p, u64p, u8p, u64p, C.c_int8, C.c_int8, C.c_int8, C.c_int8, C.c_int, C.c_int,
                                     C.POINTER(Ez), u32p, u64p, C.c_size_t, C.POINTER(C.c_float)]
        _lib = L
    return _lib


EXPORTS = ("idl_default_params idl_create idl_destroy idl_batch_alloc idl_batch_free idl_submit idl_upload idl_run_resident idl_wait "
           "idl_release idl_strerror idl_last_cuda_error idl_device_count idl_ksw2_batch idl_sweep idl_sweep_free "
           "idl_bam_open idl_bam_get_info idl_bam_close idl_bam_sweep idl_bam_fetch idl_bam_reads_free idl_bam_set_reference idl_bam_submit idl_bam_pack idl_bam_open_slice idl_device_memory idl_bam_sweep_window "
           "idl_fasta_open idl_fasta_get_info idl_fasta_copy idl_fasta_close idl_bam_set_reference_fasta").split()


class SweepIn(C.Structure):
    _fields_ = [("chrom_len", C.c_int32), ("n_reads", C.c_size_t), ("start", C.POINTER(C.c_int32)), ("stop", C.POINTER(C.c_int32)), ("flag", C.POINTER(C.c_uint16)),
                ("cigar", u32p), ("cig_off", u64p)]


class SweepOut(C.Structure):
    _fields_ = [("n_rois", C.c_size_t), ("roi_start", C.POINTER(C.c_int32)), ("roi_end", C.POINTER(C.c_int32)), ("roi_read_begin", C.POINTER(C.c_int64)),
                ("roi_n_reads", C.POINTER(C.c_int32)), ("n_read_idx", C.c_size_t), ("read_idx", C.POINTER(C.c_int64)), ("n_runs", C.c_size_t),
                ("n_evidence", C.c_size_t), ("evidence", u8p), ("ms_h2d", C.c_float), ("ms_kernels", C.c_float), ("ms_d2h", C.c_float),
                ("algorithmic_bytes", C.c_uint64), ("streamed_bytes", C.c_uint64), ("n_edge", C.c_size_t * 2)]


def sweep(chrom_len, start, stop, flag, cigar, cig_off, min_event_support=3, min_read_coverage=3, max_read_coverage=600, evidence=False, device=0):
    """idl_sweep for one target: gen_roi (src/indelope.nim:515-545) on the GPU.  Arrays are numpy (int32, int32, uint16, uint32, uint64).
    Returns a dict of numpy arrays (copies) + timings."""
    L = lib()
    L.idl_sweep.argtypes = [C.c_int, C.POINTER(SweepIn), C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.POINTER(SweepOut))]
    L.idl_sweep_free.argtypes = [C.POINTER(SweepOut)]
    a = [np.ascontiguousarray(x, dtype=t) for x, t in ((start, np.int32), (stop, np.int32), (flag, np.uint16), (cigar, np.uint32), (cig_off, np.uint64))]
    si = SweepIn(int(chrom_len), len(a[0]), a[0].ctypes.data_as(C.POINTER(C.c_int32)), a[1].ctypes.data_as(C.POINTER(C.c_int32)), a[2].ctypes.data_as(C.POINTER(C.c_uint16)),
                 a[3].ctypes.data_as(u32p), a[4].ctypes.data_as(u64p))
    out = C.POINTER(SweepOut)()
    rc = L.idl_sweep(device, C.byref(si), min_event_support, min_read_coverage, max_read_coverage, 1 if evidence else 0, C.byref(out))
    if rc != 0:
        raise IdlError("idl_sweep: %s" % L.idl_strerror(rc).decode())
    return _sweep_out(L, out, evidence)


def _sweep_out(L, out, evidence=False):
    o = out.contents
    def arr(p, n, t):
        return np.ctypeslib.as_array(p, shape=(n,)).astype(t, copy=True) if n else np.zeros(0, t)
    r = dict(roi_start=arr(o.roi_start, o.n_rois, np.int32), roi_end=arr(o.roi_end, o.n_rois, np.int32), roi_read_begin=arr(o.roi_read_begin, o.n_rois, np.int64),
             roi_n_reads=arr(o.roi_n_reads, o.n_rois, np.int32), read_idx=arr(o.read_idx, o.n_read_idx, np.int64), n_runs=int(o.n_runs),
             evidence=arr(o.evidence, o.n_evidence, np.uint8) if evidence else None, ms_h2d=o.ms_h2d, ms_kernels=o.ms_kernels, ms_d2h=o.ms_d2h,
             algorithmic_bytes=int(o.algorithmic_bytes), streamed_bytes=int(o.streamed_bytes), n_edge=(int(o.n_edge[0]), int(o.n_edge[1])))
    L.idl_sweep_free(out)
    return r


class BamInfo(C.Structure):
    _fields_ = [("file_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64), ("n_members", C.c_uint32), ("boundary_fixups", C.c_uint32), ("n_ref", C.c_int32),
                ("ref_name", C.POINTER(C.c_char_p)), ("ref_len", C.POINTER(C.c_int64)), ("header_text", C.c_void_p), ("header_len", C.c_size_t),
                ("n_records", C.c_int64), ("n_unplaced", C.c_int64), ("ref_first", C.POINTER(C.c_int64)), ("ms_h2d", C.c_float), ("ms_inflate", C.c_float),
                ("ms_parse", C.c_float), ("n_chunks", C.c_uint32)]


class BamReads(C.Structure):
    _fields_ = [("n", C.c_size_t), ("chrom", C.POINTER(C.c_int32)), ("start", C.POINTER(C.c_int32)), ("stop", C.POINTER(C.c_int32)), ("len", C.POINTER(C.c_int32)),
                ("mapq", u8p), ("flag", C.POINTER(C.c_uint16)), ("seq_off", C.POINTER(C.c_int64)), ("bases", u8p), ("quals", u8p), ("cig_off", u64p), ("cigar", u32p),
                ("ms_kernels", C.c_float), ("ms_d2h", C.c_float)]


BAM_SEQ, BAM_CIGAR = 1, 2


class BamSlice(C.Structure):
    _fields_ = [("n_ref", C.c_int32), ("ref_name", C.POINTER(C.c_char_p)), ("ref_len", C.POINTER(C.c_int64)), ("first_record", C.c_uint64), ("end_member", C.c_uint64),
                ("end_offset", C.c_uint64)]


class Bam:
    """idl_bam_*: a BAM file inflated and parsed on the GPU (SURVEY 8(f)3).  `data` = the file's bytes, or -- with `slice` = dict(ref_names, ref_len,
    first_record, end_member, end_offset) -- a run of whole BGZF members holding one target's records (idl_bam_open_slice; host.bai_target_span)."""

    def __init__(self, data, device=0, slice=None):
        L = lib()
        L.idl_bam_open_slice.argtypes = [C.c_int, C.c_char_p, C.c_size_t, C.POINTER(BamSlice), C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t]
        L.idl_bam_open.argtypes = [C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t]
        L.idl_bam_get_info.argtypes = [C.c_void_p]; L.idl_bam_get_info.restype = C.POINTER(BamInfo)
        L.idl_bam_close.argtypes = [C.c_void_p]
        L.idl_bam_sweep.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.POINTER(SweepOut))]
        L.idl_sweep_free.argtypes = [C.POINTER(SweepOut)]
        L.idl_bam_fetch.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int64), C.c_uint32, C.POINTER(C.POINTER(BamReads))]
        L.idl_bam_reads_free.argtypes = [C.POINTER(BamReads)]
        self.h = C.c_void_p()
        err = C.create_string_buffer(512)
        if slice is None:
            rc = L.idl_bam_open(device, data, len(data), C.byref(self.h), err, 512)
        else:
            n = len(slice["ref_names"])
            names = (C.c_char_p * n)(*[x.encode() for x in slice["ref_names"]])
            lens = np.ascontiguousarray(slice["ref_len"], dtype=np.int64)
            sl = BamSlice(n, names, lens.ctypes.data_as(C.POINTER(C.c_int64)), int(slice["first_record"]), int(slice["end_member"]), int(slice["end_offset"]))
            rc = L.idl_bam_open_slice(device, data, len(data), C.byref(sl), C.byref(self.h), err, 512)
        if rc != 0:
            self.h = None
            raise IdlError("idl_bam_open: %s: %s" % (L.idl_strerror(rc).decode(), err.value.decode()))
        i = L.idl_bam_get_info(self.h).contents
        self.n_ref = int(i.n_ref)
        self.ref_names = [i.ref_name[k].decode() for k in range(self.n_ref)]
        self.ref_len = [int(i.ref_len[k]) for k in range(self.n_ref)]
        self.ref_first = [int(i.ref_first[k]) for k in range(self.n_ref + 1)]
        self.header = C.string_at(i.header_text, i.header_len).decode() if i.header_len else ""
        self.n_records, self.n_unplaced = int(i.n_records), int(i.n_unplaced)
        self.info = dict(file_bytes=int(i.file_bytes), inflated_bytes=int(i.inflated_bytes), n_members=int(i.n_members), boundary_fixups=int(i.boundary_fixups),
                         ms_h2d=i.ms_h2d, ms_inflate=i.ms_inflate, ms_parse=i.ms_parse, n_chunks=int(i.n_chunks))

    def sweep(self, target, min_event_support=3, min_read_coverage=3, max_read_coverage=600, evidence=False):
        L = lib()
        out = C.POINTER(SweepOut)()
        rc = L.idl_bam_sweep(self.h, target, min_event_support, min_read_coverage, max_read_coverage, 1 if evidence else 0, C.byref(out))
        if rc != 0:
            raise IdlError("idl_bam_sweep: %s" % L.idl_strerror(rc).decode())
        return _sweep_out(L, out, evidence)

    def sweep_window(self, target, zone_lo, zone_hi, iv_beg, iv_end, min_event_support=3, min_read_coverage=3, max_read_coverage=600, evidence=False):
        """idl_bam_sweep_window: the regions of positions zone_lo .. zone_hi that overlap one of the sorted, disjoint intervals [iv_beg[k], iv_end[k]) and lie
        strictly inside the zone's inner edges; n_edge = (selected runs touching zone_lo, touching zone_hi), left out"""
        L = lib()
        i32 = C.POINTER(C.c_int32)
        L.idl_bam_sweep_window.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_size_t, i32, i32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32,
                                           C.POINTER(C.POINTER(SweepOut))]
        b = np.ascontiguousarray(iv_beg, dtype=np.int32); e = np.ascontiguousarray(iv_end, dtype=np.int32)
        out = C.POINTER(SweepOut)()
        rc = L.idl_bam_sweep_window(self.h, target, int(zone_lo), int(zone_hi), len(b), b.ctypes.data_as(i32), e.ctypes.data_as(i32), min_event_support,
                                    min_read_coverage, max_read_coverage, 1 if evidence else 0, C.byref(out))
        if rc != 0:
            raise IdlError("idl_bam_sweep_window: %s" % L.idl_strerror(rc).decode())
        return _sweep_out(L, out, evidence)

    def fetch(self, idx=None, what=BAM_SEQ | BAM_CIGAR):
        """records idx (None: all) as numpy arrays"""
        L = lib()
        out = C.POINTER(BamReads)()
        if idx is None:
            n, ip = self.n_records, None
        else:
            ia = np.ascontiguousarray(idx, dtype=np.int64); n, ip = len(ia), ia.ctypes.data_as(C.POINTER(C.c_int64))
        rc = L.idl_bam_fetch(self.h, n, ip, what, C.byref(out))
        if rc != 0:
            raise IdlError("idl_bam_fetch: %s" % L.idl_strerror(rc).decode())
        o = out.contents
        def arr(p, k, t):
            return np.ctypeslib.as_array(p, shape=(k,)).astype(t, copy=True) if k and p else np.zeros(0, t)
        r = dict(chrom=arr(o.chrom, n, np.int32), start=arr(o.start, n, np.int32), stop=arr(o.stop, n, np.int32), len=arr(o.len, n, np.int32), mapq=arr(o.mapq, n, np.uint8),
                 flag=arr(o.flag, n, np.uint16), ms_kernels=o.ms_kernels, ms_d2h=o.ms_d2h)
        if what & BAM_SEQ:
            r["seq_off"] = arr(o.seq_off, n + 1, np.int64)
            nb = int(r["seq_off"][-1]) if n else 0
            r["bases"] = arr(o.bases, nb, np.uint8); r["quals"] = arr(o.quals, nb, np.uint8)
        if what & BAM_CIGAR:
            r["cig_off"] = arr(o.cig_off, n + 1, np.uint64)
            r["cigar"] = arr(o.cigar, int(r["cig_off"][-1]) if n else 0, np.uint32)
        L.idl_bam_reads_free(out)
        return r

    def set_reference_fasta(self, target, fasta, record):
        """the sequence of one target from record `record` of a Fasta on the same device (a device-to-device copy)"""
        L = lib()
        L.idl_bam_set_reference_fasta.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]
        rc = L.idl_bam_set_reference_fasta(self.h, target, fasta.h, record)
        if rc != 0:
            raise IdlError("idl_bam_set_reference_fasta: %s" % L.idl_strerror(rc).decode())

    def set_reference(self, target, seq):
        """the sequence of one target (ASCII bytes / uint8 array, as in the FASTA) for the batches built on the device"""
        a = np.ascontiguousarray(seq, dtype=np.uint8)
        L = lib()
        L.idl_bam_set_reference.argtypes = [C.c_void_p, C.c_int32, u8p, C.c_int64]
        rc = L.idl_bam_set_reference(self.h, target, a.ctypes.data_as(u8p), len(a))
        if rc != 0:
            raise IdlError("idl_bam_set_reference: %s" % L.idl_strerror(rc).decode())

    def close(self):
        if self.h:
            lib().idl_bam_close(self.h); self.h = None

    def __del__(self):
        self.close()


class FastaInfo(C.Structure):
    _fields_ = [("file_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64), ("sequence_bytes", C.c_uint64), ("n_members", C.c_uint32), ("n_chunks", C.c_uint32),
                ("n_records", C.c_int64), ("name", C.POINTER(C.c_char_p)), ("len", C.POINTER(C.c_int64)), ("ms_h2d", C.c_float), ("ms_inflate", C.c_float),
                ("ms_parse", C.c_float), ("parse_algorithmic_bytes", C.c_uint64), ("parse_streamed_bytes", C.c_uint64)]


class Fasta:
    """idl_fasta_*: a bgzip-compressed FASTA (`data` = the file's bytes) inflated and parsed on the GPU; the sequences stay there.  IdlError for plain
    gzip, a corrupt member or a text that does not start with '>'."""

    def __init__(self, data, device=0):
        L = lib()
        L.idl_fasta_open.argtypes = [C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t]
        L.idl_fasta_get_info.argtypes = [C.c_void_p]; L.idl_fasta_get_info.restype = C.POINTER(FastaInfo)
        L.idl_fasta_copy.argtypes = [C.c_void_p, C.c_int64, u8p, C.c_size_t]
        L.idl_fasta_close.argtypes = [C.c_void_p]
        self.h = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = L.idl_fasta_open(device, data, len(data), C.byref(self.h), err, 512)
        if rc != 0:
            self.h = None
            raise IdlError("idl_fasta_open: %s: %s" % (L.idl_strerror(rc).decode(), err.value.decode()))
        i = L.idl_fasta_get_info(self.h).contents
        self.n_records = int(i.n_records)
        self.names = [i.name[k].decode("latin-1") for k in range(self.n_records)]
        self.lengths = [int(i.len[k]) for k in range(self.n_records)]
        self.info = {k: getattr(i, k) for k in ("file_bytes", "inflated_bytes", "sequence_bytes", "n_members", "n_chunks", "ms_h2d", "ms_inflate", "ms_parse",
                                                 "parse_algorithmic_bytes", "parse_streamed_bytes")}

    def sequence(self, record):
        """one record's sequence copied to the host (uint8 array)"""
        out = np.empty(self.lengths[record], dtype=np.uint8)
        rc = lib().idl_fasta_copy(self.h, record, out.ctypes.data_as(u8p), len(out))
        if rc != 0:
            raise IdlError("idl_fasta_copy: %s" % lib().idl_strerror(rc).decode())
        return out

    def close(self):
        if self.h:
            lib().idl_fasta_close(self.h); self.h = None

    def __del__(self):
        self.close()


def _roi_args(roi_chrom, roi_start, roi_end, roi_n_reads, read_idx):
    a = [np.ascontiguousarray(x, dtype=t) for x, t in ((roi_chrom, np.int32), (roi_start, np.int32), (roi_end, np.int32), (roi_n_reads, np.int32), (read_idx, np.int64))]
    i32 = C.POINTER(C.c_int32)
    return a, (len(a[0]), a[0].ctypes.data_as(i32), a[1].ctypes.data_as(i32), a[2].ctypes.data_as(i32), a[3].ctypes.data_as(i32), a[4].ctypes.data_as(C.POINTER(C.c_int64)))


class Context:
    """one per GPU (idl_create / idl_destroy)"""

    def __init__(self, device=0, params=None, **kw):
        self.params = params if params is not None else default_params(**kw)
        self.h = C.c_void_p()
        rc = lib().idl_create(device, C.byref(self.params), C.byref(self.h))
        if rc != 0:
            self.h = None
            raise IdlError("idl_create: %s" % lib().idl_strerror(rc).decode())

    def _check(self, rc, what):
        if rc != 0:
            raise IdlError("%s: %s (%s)" % (what, lib().idl_strerror(rc).decode(), lib().idl_last_cuda_error(self.h).decode()))

    def batch_alloc(self, max_regions, max_reads, max_seq_bases, max_ref_bases):
        b = C.POINTER(Batch)()
        self._check(lib().idl_batch_alloc(self.h, max_regions, max_reads, max_seq_bases, max_ref_bases, C.byref(b)), "idl_batch_alloc")
        return b

    def batch_free(self, b):
        lib().idl_batch_free(self.h, b)

    def submit(self, batch):
        t = C.c_uint64()
        self._check(lib().idl_submit(self.h, batch, C.byref(t)), "idl_submit")
        return t.value

    def bam_submit(self, bam, roi_chrom, roi_start, roi_end, roi_n_reads, read_idx, ordinal_base=0):
        """idl_bam_submit: the batch of these regions is built on the device from the resident BAM and run; returns the ticket"""
        L = lib()
        i32 = C.POINTER(C.c_int32)
        L.idl_bam_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, i32, i32, i32, i32, C.POINTER(C.c_int64), C.c_uint32, u64p]
        keep, args = _roi_args(roi_chrom, roi_start, roi_end, roi_n_reads, read_idx)
        t = C.c_uint64()
        self._check(L.idl_bam_submit(self.h, bam.h, *args, ordinal_base, C.byref(t)), "idl_bam_submit")
        return t.value

    def bam_pack(self, bam, roi_chrom, roi_start, roi_end, roi_n_reads, read_idx, batch, ordinal_base=0):
        """idl_bam_pack: the same batch copied into a host idl_batch (from batch_alloc)"""
        L = lib()
        i32 = C.POINTER(C.c_int32)
        L.idl_bam_pack.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, i32, i32, i32, i32, C.POINTER(C.c_int64), C.c_uint32, C.POINTER(Batch)]
        keep, args = _roi_args(roi_chrom, roi_start, roi_end, roi_n_reads, read_idx)
        self._check(L.idl_bam_pack(self.h, bam.h, *args, ordinal_base, batch), "idl_bam_pack")

    def upload(self, batch):
        self._check(lib().idl_upload(self.h, batch), "idl_upload")

    def run_resident(self, batch):
        t = C.c_uint64()
        self._check(lib().idl_run_resident(self.h, batch, C.byref(t)), "idl_run_resident")
        return t.value

    def wait(self, ticket):
        r = C.POINTER(Results)()
        self._check(lib().idl_wait(self.h, ticket, C.byref(r)), "idl_wait")
        return r

    def release(self, ticket):
        self._check(lib().idl_release(self.h, ticket), "idl_release")

    def ksw2_batch(self, queries, targets, match=1, mismatch=-2, gapo=4, gape=1, w=-1, zdrop=-1):
        """queries/targets: lists of uint8 code arrays (0..4). Returns (list of field dicts, list of cigar tuples, kernel ms)"""
        n = len(queries)
        qo = np.zeros(n + 1, dtype=np.uint64); to = np.zeros(n + 1, dtype=np.uint64)
        qo[1:] = np.cumsum([len(q) for q in queries]); to[1:] = np.cumsum([len(t) for t in targets])
        qa = np.ascontiguousarray(np.concatenate([np.asarray(q, dtype=np.uint8) for q in queries] + [np.zeros(1, np.uint8)]))
        ta = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.uint8) for t in targets] + [np.zeros(1, np.uint8)]))
        out = (Ez * n)()
        cap = int(qo[-1] + to[-1]) + 8 * n + 16
        cig = np.zeros(cap, dtype=np.uint32); coff = np.zeros(n, dtype=np.uint64)
        ms = C.c_float()
        self._check(lib().idl_ksw2_batch(self.h, n, qa.ctypes.data_as(u8p), qo.ctypes.data_as(u64p), ta.ctypes.data_as(u8p), to.ctypes.data_as(u64p),
                                         C.c_int8(match), C.c_int8(mismatch), C.c_int8(gapo), C.c_int8(gape), w, zdrop, out, cig.ctypes.data_as(u32p),
                                         coff.ctypes.data_as(u64p), cap, C.byref(ms)), "idl_ksw2_batch")
        names = "max zdropped max_q max_t mqe mqe_t mte mte_q score n_cigar".split()
        fields = [{k: getattr(out[i], k) for k in names} for i in range(n)]
        cigs = [tuple(int(x) for x in cig[int(coff[i]):int(coff[i]) + max(out[i].n_cigar, 0)]) for i in range(n)]
        extra = [dict(status=out[i].status, cells=out[i].cells) for i in range(n)]
        return fields, cigs, extra, ms.value

    def close(self):
        if getattr(self, "h", None):
            lib().idl_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()
