"""Host-side mirror of the reference's calling loop over the two native libraries.

    for r in gen_roi(...): for v in callsemble(r, ...): dedup; echo v        (src/indelope.nim:601-608)

becomes: pack regions into pinned batches -> idl_submit (async, one lane per stream) -> idl_wait -> filter cascade +
VCF text on the host.  Regions keep their emission order (batches are contiguous slices, records are written in
ticket order), so the order-dependent dedup sees the same sequence as the reference's single loop.
"""
import ctypes as C

import numpy as np

from . import cuda, host
from .abi import default_params


def plan_batches(rois, lo, hi, max_reads=400_000, max_regions=20_000):
    """contiguous slices [a, b) of the region list, bounded by reads and regions per batch"""
    n = np.ctypeslib.as_array(rois.c.roi_n_reads, shape=(rois.n_rois,)) if rois.n_rois else np.zeros(0, np.int32)
    out, a, acc = [], lo, 0
    for k in range(lo, hi):
        if k > a and (acc + int(n[k]) > max_reads or k - a >= max_regions):
            out.append((a, k)); a, acc = k, 0
        acc += int(n[k])
    if hi > a:
        out.append((a, hi))
    return out


def gpu_rois(ds, min_reads=3, max_read_coverage=600, device=0, timings=None):
    """gen_roi for every target of a dataset ON THE GPU (idl_sweep, SURVEY.md 8(f)4): the same regions and record lists as
    ds.sweep(min_reads) -- src/indelope.nim:515-545,601-602 with min_event_support = max(3, min_reads - 2) -- as a host.Rois"""
    base = host.Rois(host.lib().idlh_sweep(ds.h, 255, 1 << 30, 1 << 30), ds)  # no regions: just the record arrays of the dataset
    a = dict(base.arrays())
    chrom, rs, re, nr, idx = [], [], [], [], []
    for c in range(ds.n_chroms):
        cr = ds.chrom_reads(c)
        r = cuda.sweep(cr["chrom_len"], cr["start"], cr["stop"], cr["flag"], cr["cigar"], cr["cig_off"], min_event_support=max(3, min_reads - 2),
                       min_read_coverage=min_reads, max_read_coverage=max_read_coverage, device=device)
        chrom.append(np.full(len(r["roi_start"]), c, np.int32)); rs.append(r["roi_start"]); re.append(r["roi_end"]); nr.append(r["roi_n_reads"])
        idx.append(r["read_idx"] + cr["first_read"])
        if timings is not None:
            timings.append({k: r[k] for k in ("ms_h2d", "ms_kernels", "ms_d2h", "algorithmic_bytes", "streamed_bytes", "n_runs")})
    a["roi_chrom"] = np.concatenate(chrom); a["roi_start"] = np.concatenate(rs); a["roi_stop"] = np.concatenate(re); a["roi_n_reads"] = np.concatenate(nr)
    a["read_idx"] = np.concatenate(idx)
    a["roi_read_begin"] = np.concatenate([[0], np.cumsum(a["roi_n_reads"])[:-1]]).astype(np.int64) if len(a["roi_n_reads"]) else np.zeros(0, np.int64)
    out = host.Rois(arrays=a)
    out._keep = (base, ds)  # the arrays are views of the dataset's memory
    return out


class Caller:
    """`indelope --min-reads M --min-contig-len C --min-event-len E` over regions, on one GPU"""

    def __init__(self, device=0, min_reads=3, min_ctg_len=73, min_event_len=4, **kw):
        self.params = default_params(min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len, **kw)
        self.ctx = cuda.Context(device, self.params)
        self._batches = {}

    def _batch_for(self, lane, sizes):
        """pinned batch per lane, grown on demand"""
        cur = self._batches.get(lane)
        need = (sizes[0], sizes[1], sizes[2], sizes[3])
        if cur is None or any(n > c for n, c in zip(need, cur[1])):
            if cur is not None:
                self.ctx.batch_free(cur[0])
            cap = tuple(int(x * 1.25) + 64 for x in need)
            cur = (self.ctx.batch_alloc(*cap), cap)
            self._batches[lane] = cur
        return cur[0]

    def call(self, rois, lo=0, hi=None, dump_level=0, max_reads=400_000, timings=None, dedup=True):
        """returns (vcf record text, dump text). `timings` (list) receives one dict per batch.  dedup=False leaves the
        order-dependent dedup to the caller (interval shards are merged first, see indelope_b200.shard)."""
        hi = rois.n_rois if hi is None else hi
        writer = host.VcfWriter(dedup=dedup)
        plans = plan_batches(rois, lo, hi, max_reads=max_reads)
        n_lanes = self.params.n_streams
        vcf, dump = [], []
        inflight = []

        def drain():
            a, b, t = inflight.pop(0)
            res = self.ctx.wait(t)
            v, d = writer.records(rois, a, self.params, res, dump_level)
            if timings is not None:
                r = res.contents
                timings.append({k: getattr(r, k) for k in ("ms_h2d", "ms_assemble", "ms_align", "ms_genotype", "ms_al", "ms_d2h", "ms_total", "n_regions",
                                                           "n_contigs", "n_alns", "n_events", "offsets_tested", "dp_cells_a", "dp_cells_b", "dp_a", "dp_b",
                                                           "kmer_reads", "kmer_bytes", "al_events", "kernel_launches", "pool_retries")})
            self.ctx.release(t)
            vcf.append(v); dump.append(d)

        for i, (a, b) in enumerate(plans):
            if len(inflight) >= n_lanes:
                drain()
            nr, sb, rb = rois.pack_size(a, b, self.params)
            batch = self._batch_for(i % n_lanes, (b - a, nr, sb, rb))
            rois.pack(a, b, self.params, batch)
            inflight.append((a, b, self.ctx.submit(batch)))
        while inflight:
            drain()
        self.status_counts = writer.status_counts()  # regions per IDL_RS_* bit of the last call (warnings went to stderr)
        return "".join(vcf), "".join(dump)

    def close(self):
        for b, _ in self._batches.values():
            self.ctx.batch_free(b)
        self._batches = {}
        self.ctx.close()


def call_bam(fasta, bam, device=0, min_reads=3, min_ctg_len=73, min_event_len=4, max_reads=400_000, by_target=False, timings=None, regions=None, bed=None, **kw):
    """`indelope --gpu-decode [options] <fasta> <bam>` in process: the VCF (header + records) with everything in front of callsemble on the
    device as well -- BGZF inflate and record parse (idl_bam_open), gen_roi per target (idl_bam_sweep, src/indelope.nim:515-545,601-602), the
    batches built from the resident records (idl_bam_submit).  The host reads the two files and writes the VCF text.
    regions (list of `chr[:beg[-end]]`, 1-based, inclusive) and / or bed (a BED file, 0-based, half open): `indelope -r ... -R ...` -- only the regions of
    interest of the whole-file run that overlap them, from just the BGZF members that hold them (idl_bam_open_slice, idl_bam_sweep_window; needs the
    index).  `timings` then also receives one dict per target with slices, retries and bytes read and decoded.  ValueError for a bad region or BED line.
    by_target: the file is not decoded as a whole but target by target, through the same loop with every target whole as its interval -- for files
    that do not fit in device memory; needs the index.
    A FASTA compressed with bgzip is inflated and parsed on the device (cuda.Fasta); the batches take the targets' sequences from there."""
    if regions or bed:
        by_target = True
    fa_dev, record_of = None, None
    with open(fasta, "rb") as f:
        if f.read(2) == b"\x1f\x8b":
            f.seek(0)
            fa_dev = cuda.Fasta(f.read(), device=device)
    if fa_dev is not None:
        ref = host.Dataset.from_sequences(fa_dev.names, [fa_dev.sequence(r) for r in range(fa_dev.n_records)])
    if by_target:
        if fa_dev is not None:
            ref.set_bam_targets(bam)
            names, seqs = ref.sequences()
            keep = (ref, fa_dev)
        else:
            st = host.Stream(fasta, bam)      # parses the BAM header and orders the FASTA's sequences after it; no record is read through it
            tg = st.targets()
            ta = tg.arrays()
            names, seqs = ta["chrom_names"], ta["chrom_seqs"]
            keep = (st, tg)
        ref_len = [len(x) for x in seqs]
    else:
        if fa_dev is None:
            ref = host.Dataset.load_fasta(fasta)
        data = open(bam, "rb").read()
        whole = cuda.Bam(data, device=device)
        ref.set_targets(whole.ref_names, whole.ref_len)
        names, seqs = ref.sequences()
        keep = (ref, fa_dev)
    if fa_dev is not None:   # each target's record: the first of its name, as set_targets takes it
        first = {}
        for r, nm in enumerate(fa_dev.names):
            first.setdefault(nm, r)
        record_of = [first[nm] for nm in names]
    if by_target:
        selected = host.parse_regions(names, ref_len, regions, bed) if regions or bed else [[(0, n)] for n in ref_len]
        if names:
            host.bai_target_span(bam, 0)      # IOError without the index, before anything runs
    caller = Caller(device, min_reads=min_reads, min_ctg_len=min_ctg_len, min_event_len=min_event_len, **kw)
    writer = host.VcfWriter()
    empty = dict(start=[], stop=[], mapq=[], flag=[], len=[], seq_off=[], bases=[], quals=[])
    out = [host.Rois(arrays=dict(empty, roi_chrom=[], roi_start=[], roi_stop=[], roi_read_begin=[], roi_n_reads=[], read_idx=[], chrom_names=names, chrom_seqs=seqs)).header()]
    done = [0]
    sweep_args = dict(min_event_support=max(3, min_reads - 2), min_read_coverage=min_reads, max_read_coverage=600)

    def call_resident(b, c, r, first=0):
        """regions [first, n) of one sweep of b through idl_bam_submit, records appended to out"""
        n = len(r["roi_start"]) - first
        if n <= 0:
            return
        chrom = np.full(n, c, np.int32)
        rs, re, nr = r["roi_start"][first:], r["roi_end"][first:], r["roi_n_reads"][first:]
        idx = r["read_idx"][int(r["roi_read_begin"][first]):]
        begin = np.concatenate([[0], np.cumsum(nr)]).astype(np.int64)
        rois = host.Rois(arrays=dict(empty, roi_chrom=chrom, roi_start=rs, roi_stop=re, roi_read_begin=begin[:-1], roi_n_reads=nr, read_idx=idx, chrom_names=names, chrom_seqs=seqs))
        if fa_dev is not None:
            b.set_reference_fasta(c, fa_dev, record_of[c])
        else:
            b.set_reference(c, seqs[c])
        inflight = []

        def drain():
            lo, t = inflight.pop(0)
            res = caller.ctx.wait(t)
            v, _ = writer.records(rois, lo, caller.params, res, 0)
            if timings is not None:
                timings.append({k: getattr(res.contents, k) for k in ("ms_assemble", "ms_align", "ms_genotype", "ms_al", "n_regions", "n_events")})
            caller.ctx.release(t); out.append(v)
        for lo, hi in plan_batches(rois, 0, n, max_reads=max_reads):
            if len(inflight) >= caller.params.n_streams:
                drain()
            inflight.append((lo, caller.ctx.bam_submit(b, chrom[lo:hi], rs[lo:hi], re[lo:hi], nr[lo:hi], idx[begin[lo]:begin[hi]], ordinal_base=done[0] + lo)))
        while inflight:
            drain()
        done[0] += n

    def call_target_regions(c, ivs):
        """the slices of one target's intervals, grown until no selected region touches an inner zone edge (indelope_main.cpp run_sliced)"""
        stats = dict(target=c, intervals=len(ivs), slices=0, retries=0, bytes_read=0, bytes_decoded=0, regions=0)
        todo = []
        for b0, e0 in ivs:
            w0, w1 = ((b0 - 1) >> 14) if b0 > 0 else 0, ((e0 - 1) >> 14) + 1
            if todo and w0 <= todo[-1][1]:
                todo[-1] = [todo[-1][0], max(todo[-1][1], w1), todo[-1][2] + [(b0, e0)], None]
            else:
                todo.append([w0, w1, [(b0, e0)], None])
        for s in todo:
            s[3] = host.bai_region_run(bam, c, s[0], s[1])
        last_end = -1
        while todo:
            w0, w1, iv, run = todo.pop(0)
            while todo and not run["empty"] and not todo[0][3]["empty"] and todo[0][3]["file_begin"] <= run["file_end"]:
                n = todo.pop(0); w1 = max(w1, n[1]); iv = iv + n[2]
                run = host.bai_region_run(bam, c, w0, w1)
            if run["empty"]:
                if not run["to_end"]:
                    stats["retries"] += 1
                    todo.insert(0, [w0, w1 + 1, iv, host.bai_region_run(bam, c, w0, w1 + 1)])
                continue
            with open(bam, "rb") as f:
                f.seek(run["file_begin"]); data = f.read(run["file_end"] - run["file_begin"])
            b = cuda.Bam(data, device=device, slice=dict(ref_names=names, ref_len=ref_len, first_record=run["first_record"], end_member=run["end_member"],
                                                         end_offset=run["end_offset"]))
            try:
                stats["slices"] += 1; stats["bytes_read"] += len(data); stats["bytes_decoded"] += b.info["inflated_bytes"]
                zone_hi = ref_len[c] if run["to_end"] else int(b.fetch([b.n_records - 1], what=0)["start"][0]) - 1
                if zone_hi < run["zone_lo"] or zone_hi < iv[-1][1] - 1:
                    stats["retries"] += 1
                    todo.insert(0, [w0, w1 + 1, iv, host.bai_region_run(bam, c, w0, w1 + 1)])
                    continue
                r = b.sweep_window(c, run["zone_lo"], zone_hi, [x[0] for x in iv], [x[1] for x in iv], **sweep_args)
                if r["n_edge"][0] or r["n_edge"][1]:
                    stats["retries"] += 1
                    w0, w1 = w0 - (1 if r["n_edge"][0] else 0), w1 + (1 if r["n_edge"][1] else 0)
                    todo.insert(0, [w0, w1, iv, host.bai_region_run(bam, c, w0, w1)])
                    continue
                first = int(np.searchsorted(r["roi_start"], last_end, side="right"))   # regions an earlier slice (before this one grew left) called
                call_resident(b, c, r, first)
                stats["regions"] += len(r["roi_start"]) - first
                if len(r["roi_start"]) > first:
                    last_end = int(r["roi_end"][-1])
            finally:
                b.close()
        if timings is not None:
            timings.append(stats)

    try:
        for c, name in enumerate(names):
            if name == "hs37d5" or name.startswith("GL"):   # skippable targets, src/indelope.nim:41-42
                continue
            if not by_target:
                call_resident(whole, c, whole.sweep(c, **sweep_args))
            elif selected[c]:
                call_target_regions(c, selected[c])
        caller.status_counts = writer.status_counts()
    finally:
        caller.close()
        if not by_target:
            whole.close()
    del keep
    return "".join(out)
