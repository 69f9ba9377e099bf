#!/usr/bin/env python
"""bench.py -- throughput of indelope's per-region calling path on B200 (see DESIGN.md "Measurement").

  python bench.py --gpus 1 --steps 80 --warmup 3                   # this repo's CUDA path, chr1 workload (BASELINE config 3)
  python bench.py --impl reference --gpus 1 --steps 2 --warmup 1   # the reference algorithm on the host cores (CPU oracle)
  python bench.py --workload wgs --gpus N                          # BASELINE config 5: ONE 24-contig genome, interval-sharded (strong scaling)
  python bench.py --workload {pr1,exome,panel500,panel500_lowerr}  # the other configs (profiles/r02_bench_<cfg>.json)

A "step" is one pass of the hot path (assemble -> align -> k-mer genotype -> AL fallback) over one workload of synthetic candidate
regions.  Weak scaling (default): rank r of N builds its own interval shard (seed + 1000 r) of the same size; value = regions of all
ranks / max-over-ranks step time.  Strong scaling (--workload wgs): the 24 contigs of one genome are dealt to the ranks in contiguous
blocks, every rank calls its block, the records are gathered on rank 0 in rank order and the order-dependent dedup of
src/indelope.nim:604-608 runs over the merged text -- inside the timed end-to-end region.  Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OUT = sys.stdout
CALL = dict(min_reads=5, min_ctg_len=73, min_event_len=5)  # `indelope --min-event-len 5 --min-reads 5` (BASELINE.json configs[0])
WGS_CONTIGS = 24


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=80, help="timed steps (80 x ~40 ms: a timed region of seconds, so that clocks and power settle)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="chr1", help="key of indelope_b200.host.CONFIGS")
    ap.add_argument("--mode", default="auto", choices=["auto", "weak", "strong"], help="auto: strong for --workload wgs, weak otherwise")
    ap.add_argument("--scale", type=float, default=1.0, help="scale the number of planted events (tests)")
    ap.add_argument("--cpu-sample", type=int, default=40000, help="regions timed by the cpu_baseline leg (about 15 s of one core)")
    ap.add_argument("--no-bam-leg", action="store_true", help="skip the leg that starts from a BAM resident on the device (idl_bam_open + idl_bam_submit; N=1 only: it writes the workload as a BAM first)")
    ap.add_argument("--e2e-batches", type=int, default=2, help="batches per step in the end-to-end leg (measured: 2 -> 41.6 ms per step, 3 -> 42.7, 4 -> 42.7: smaller batches leave the persistent kernels too few tasks per warp)")
    ap.add_argument("--verify", type=int, default=1, help="strong mode: compare the merged VCF with the oracle's once after timing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after timing, write what the timed path computed in its last step (rank 0) as DIR/<name>.npy, "
                    "float32/float64, at most 64 MB in all.  Weak mode: the result tables of the end-to-end leg (idl_submit / idl_wait, whose results "
                    "reach the caller), not of the resident leg behind `value`, which copies back counters only; they are copied after that leg's "
                    "timed window closes.  Strong mode and --impl reference: the merged VCF text")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def scaling_mode(args):
    return ("strong" if args.workload == "wgs" else "weak") if args.mode == "auto" else args.mode


def build_workload(name, rank, world, scale, mode):
    from indelope_b200 import host
    cfg = dict(host.CONFIGS[name])
    cfg["n_events"] = max(1, int(cfg["n_events"] * scale))
    if mode == "strong":
        # one genome of WGS_CONTIGS contigs (every contig has its own random stream): rank r builds and calls the contigs of its block
        per = max(1, WGS_CONTIGS // world)
        cfg["n_chroms"] = per; cfg["chrom_first"] = rank * per
    else:
        cfg["seed"] = cfg["seed"] + 1000 * rank
    ds = host.Dataset(**cfg)
    rois = ds.sweep(min_reads=CALL["min_reads"])
    return cfg, ds, rois


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)"""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        pw = []
        for s in self.samples:
            try:
                pw.append(float(s[2]))
            except ValueError:
                pass
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(self.samples),
                "power_w_max": max(pw) if pw else None}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)", d.get("sm_max_mhz", 1965.0)
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def cpu_model():
    try:
        for l in open("/proc/cpuinfo"):
            if l.startswith("model name"):
                return l.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def oracle_build_flags():
    try:
        mk = open(os.path.join(ROOT, "oracle", "Makefile")).read()
        fl = {k: l.split("=", 1)[1].strip() for l in mk.splitlines() for k in ("CFLAGS", "CXXFLAGS") if l.startswith(k)}
        return "g++ %s (oracle.cpp), gcc %s (ksw2_lane.c), gcc -O2 (the reference's ksw2_extz2_sse.c, SSE2, oracle/_ref)" % (fl.get("CXXFLAGS", "?"), fl.get("CFLAGS", "?"))
    except OSError:
        return "unknown"


def run_oracle(rois, n_regions, n_threads, raw=False):
    """CPU restatement of the reference (oracle/), the reference's own ksw2 C when oracle/_ref was built"""
    from oracle import pyoracle as orc
    a = rois.arrays()
    n = min(n_regions, rois.n_rois)
    sub = dict(a)
    for k in ("roi_chrom", "roi_start", "roi_stop", "roi_read_begin", "roi_n_reads"):
        sub[k] = a[k][:n]
    use_ref = orc.have_ref()
    _, vcf, cnt = orc.call(sub, use_ref_ksw2=use_ref, dump_level=32 if raw else 0, n_threads=n_threads, **CALL)
    return n, int(sub["roi_n_reads"].sum()), cnt, use_ref, vcf


def workload_name(args, cfg, mode):
    if mode == "strong":
        return "%s: one genome of %d contigs x %.0f Mb, %d planted events per contig, %gx %d bp reads simulated around events (locus_only=%d), contigs dealt to the ranks in blocks, indelope --min-event-len 5 --min-reads 5" % (
            args.workload, WGS_CONTIGS, cfg["chrom_len"] / 1e6, cfg["n_events"], cfg["coverage"], cfg["read_len"], cfg.get("locus_only", 0))
    return "%s: %d planted events on a %.0f Mb contig, %gx %d bp reads simulated around events (locus_only=%d), indelope --min-event-len 5 --min-reads 5" % (
        args.workload, cfg["n_events"], cfg["chrom_len"] / 1e6, cfg["coverage"], cfg["read_len"], cfg.get("locus_only", 0))


def config_of(args, cfg, mode, rois):
    """the same dict in both arms: it names the workload, not the implementation"""
    return {"workload": workload_name(args, cfg, mode), "scaling": mode, "regions_per_gpu": rois.n_rois, "reads_per_gpu": rois.total_reads(),
            "sharding": "contiguous blocks of contigs per rank, records gathered in rank order, dedup after the merge, no data-path collective" if mode == "strong"
            else "one interval shard per rank (seed + 1000 rank), no collective"}


def dedup_text(text):
    """independent restatement of src/indelope.nim:604-608 for the checker: drop a record equal in CHROM, POS, REF, ALT to one of the last two emitted"""
    out, l1, l2 = [], None, None
    for line in text.splitlines():
        f = line.split("\t", 5)
        k = (f[0], f[1], f[3], f[4])
        if k == l1 or k == l2:
            continue
        out.append(line); l2, l1 = l1, k
    return "".join(l + "\n" for l in out)


DUMP_BYTES = 64 << 20                           # --dump-outputs writes at most this much
DUMP_SHARE = (DUMP_BYTES - (1 << 16)) // 6      # per table: six tables and a few small files
NO_EVENTS = 0xFFFFFFFF                          # IDL_NO_EVENTS


def dump_table(out, name, n, width, itemsize, gather, share=None):
    """out[name] = gather(rows) for all n rows of a table, or for a fixed, seeded sample of them when the table would take more than
    `share` bytes (DUMP_SHARE by default); the sampled row numbers go to out[name + "_rows"]"""
    share = DUMP_SHARE if share is None else share
    rows = np.arange(n)
    if n * width * itemsize > share:
        rows = np.unique(np.random.default_rng(0).integers(0, n, share // (width * itemsize + 8)))
        out[name + "_rows"] = rows.astype(np.float64)
    out[name] = gather(rows)


def dump_text(text):
    out = {}
    b = np.frombuffer(text, dtype=np.uint8)
    dump_table(out, "vcf", len(b), 1, 4, lambda rows: b[rows].astype(np.float32), share=DUMP_BYTES - (1 << 16))   # the only table
    return out


def _ragged(offsets, lengths, pos):
    """positions `pos` in the concatenation of the blocks [offsets[i], offsets[i] + lengths[i]) -> indices into the array holding the blocks"""
    ends = np.cumsum(lengths)
    i = np.searchsorted(ends, pos, side="right")
    return offsets[i] + pos - (ends[i] - lengths[i])


def result_tables(r):
    """host copies of the tables of one ticket (idl_results), taken before its release"""
    from indelope_b200 import abi

    def table(ptr, n, t):
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(t)), (n,)).copy() if n else np.zeros(0, np.dtype(t))
    return {"reg": table(r.region, r.n_regions, abi.RegionResult), "ctg": table(r.contig, r.n_contigs, abi.ContigResult),
            "aln": table(r.aln, r.n_alns, abi.AlnResult), "ev": table(r.event, r.n_events, abi.EventResult),
            "cig": table(r.cigar, r.n_cigar_ops, C.c_uint32), "seq": table(r.contig_seq, r.n_contig_bases, C.c_uint8)}


# fields that index another table of the same ticket
LINKS = {("reg", "contig_begin"): "ctg", ("ctg", "seq_off"): "seq", ("ctg", "region"): "reg", ("ctg", "aln"): "aln", ("aln", "region"): "reg",
         ("aln", "contig"): "ctg", ("aln", "cigar_off"): "cig", ("aln", "event_begin"): "ev", ("ev", "aln"): "aln"}


def merge_tables(parts):
    """the tables of a step's batches, in batch order, as one set of int64 columns: indices are moved past the rows of the batches
    before (-1 and IDL_NO_EVENTS stay); a uint64 k-mer code keeps its 64 bits"""
    m, at = {}, dict.fromkeys(("reg", "ctg", "aln", "ev", "cig", "seq"), 0)
    for p in parts:
        for t in ("reg", "ctg", "aln", "ev"):
            for f in p[t].dtype.names:
                v = p[t][f].astype(np.int64)
                if (t, f) in LINKS:
                    v = np.where((v < 0) | (v == NO_EVENTS), v, v + at[LINKS[t, f]])
                m.setdefault(t, {}).setdefault(f, []).append(v)
        for t in ("cig", "seq"):
            m.setdefault(t, []).append(p[t])
        for t in at:
            at[t] += len(p[t])
    return {t: {f: np.concatenate(v) for f, v in c.items()} if isinstance(c, dict) else np.concatenate(c) for t, c in m.items()}


def _cols(t, names, rows):
    return np.stack([t[f][rows] for f in names], axis=1).astype(np.float64).reshape(len(rows), len(names))


def dump_results(parts):
    """the result tables of a step's tickets (result_tables, in batch order) in the order a caller reads them: the regions, the contigs of
    each region, the alignment of each contig that has one, the CIGAR ops and the event records of each alignment, the bases of each
    contig.  The device hands out contig, alignment, CIGAR, event and base slots in completion order, so slot offsets are left out and
    references between tables are indices in that order: two runs, or two builds, compare row for row.  int32/uint32 fields are exact
    in float64, a uint64 k-mer code is split into two 32-bit halves, bases (ASCII) go to float32."""
    from indelope_b200 import abi
    m = merge_tables(parts)
    reg, ctg, aln, ev, cig, seq = (m[k] for k in ("reg", "ctg", "aln", "ev", "cig", "seq"))

    n_ctg = np.maximum(reg["n_contigs"], 0)
    order = _ragged(reg["contig_begin"], n_ctg, np.arange(n_ctg.sum()))
    con = {f: v[order] for f, v in ctg.items()}
    has = con["aln"] >= 0
    con["aln_index"] = np.where(has, np.cumsum(has) - 1, -1)
    al = {f: v[con["aln"][has]] for f, v in aln.items()}
    canon_ctg = np.full(len(ctg["start"]), -1, dtype=np.int64)
    canon_ctg[order] = np.arange(len(order))
    al["contig_index"] = canon_ctg[al["contig"]]
    canon_aln = np.full(len(aln["region"]), -1, dtype=np.int64)
    canon_aln[con["aln"][has]] = np.arange(int(has.sum()))
    n_cig = np.where(al["status"] & abi.RS_CIGAR_OVERFLOW, 0, np.maximum(al["n_cigar"], 0))  # an overflowed CIGAR was not written
    n_ev = np.where(al["event_begin"] == NO_EVENTS, 0, np.maximum(al["n_events"], 0))

    out = {"counts": np.array([len(reg["status"]), len(ctg["start"]), len(aln["region"]), len(ev["aln"]), len(cig), len(seq)], dtype=np.float64)}
    f = ["status", "n_contigs_pre", "n_contigs"]
    dump_table(out, "regions", len(reg["status"]), len(f), 8, lambda rows, f=f: _cols(reg, f, rows))
    f = ["start", "nreads", "len", "region", "aln_index"]
    dump_table(out, "contigs", len(order), len(f), 8, lambda rows, f=f: _cols(con, f, rows))
    f = "region ref_len max zdropped max_q max_t mqe mqe_t mte mte_q score n_cigar n_cigar_trunc n_events status contig_index".split()
    dump_table(out, "alignments", int(has.sum()), len(f), 8, lambda rows, f=f: _cols(al, f, rows))
    dump_table(out, "cigar", int(n_cig.sum()), 1, 8, lambda rows: cig[_ragged(al["cigar_off"], n_cig, rows)].astype(np.float64)[:, None])
    f = [n for n, _ in abi.EventResult._fields_ if n not in ("aln", "ref_code", "alt_code")]

    def events(rows):   # the alignment's index, the fields, the two k-mer codes as (high, low) halves
        e = {k: v[_ragged(al["event_begin"], n_ev, rows)] for k, v in ev.items()}
        e["aln_index"] = canon_aln[e["aln"]]
        for k in ("ref_code", "alt_code"):
            e[k + "_hi"], e[k + "_lo"] = (e[k] >> 32) & 0xFFFFFFFF, e[k] & 0xFFFFFFFF
        return _cols(e, ["aln_index"] + f + ["ref_code_hi", "ref_code_lo", "alt_code_hi", "alt_code_lo"], np.arange(len(rows)))
    dump_table(out, "events", int(n_ev.sum()), len(f) + 5, 8, events)
    dump_table(out, "contig_bases", int(con["len"].sum()), 1, 4, lambda rows: seq[_ragged(con["seq_off"], con["len"], rows)].astype(np.float32))
    return out


def write_dump(path, out):
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main_reference(args, rank, world):
    if rank != 0:
        return
    mode = scaling_mode(args)
    cfg, ds, rois = build_workload(args.workload, 0, world, args.scale, mode)
    cores = os.cpu_count() or 1
    sample = rois.n_rois  # every region of rank 0's share of the workload, every step
    for _ in range(args.warmup):
        run_oracle(rois, min(sample, 2000), cores)
    t0 = time.time(); regions = reads = 0
    for _ in range(args.steps):
        n, nr, cnt, use_ref, vcf = run_oracle(rois, sample, cores)
        regions += n; reads += nr
    dt = time.time() - t0
    if args.dump_outputs:
        write_dump(args.dump_outputs, dump_text(vcf.encode()))
    val = regions / dt
    line = {
        "impl": "reference", "metric": "regions_per_s", "value": val, "unit": "regions/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": mode, "vs_baseline": None, "dtype": "int8/int32/u64", "data": "synthetic",
        "reads_per_s": reads / dt,
        "config": config_of(args, cfg, mode, rois),
        "cpu_baseline": {"value": val, "unit": "regions/s", "cores": cores, "kind": "port", "cpu": cpu_model(), "build": oracle_build_flags(),
                         "sample": "all %d regions of rank 0's share of the workload per step, %d threads over regions; the Nim binary cannot be built here (no nim/hts-nim/htslib), "
                                   "so this is the CPU oracle restating src/contig.nim + src/indelope.nim:157-428%s" % (
                                       sample, cores, " calling the reference's own ksw2_extz2_sse.c compiled unmodified (oracle/_ref)" if use_ref else " with its own lane-exact ksw2")},
        "e2e": {"value": val, "unit": "regions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=OUT, flush=True)


STAGES = ("ms_assemble", "ms_align", "ms_genotype", "ms_al")
KEYS = STAGES + ("ms_total", "offsets_tested", "dp_cells_a", "dp_cells_b", "dp_a", "dp_b", "kmer_reads", "kmer_bytes", "al_events", "kernel_launches", "n_contigs",
                 "n_alns", "n_events")


def main():
    args = parse()
    # rank 0 prints ONE JSON line on stdout: keep the real stdout aside and point fd 1 at stderr, so that nothing a native
    # library prints there (NCCL writes its version banner to stdout) lands next to it
    global OUT
    sys.stdout.flush()
    OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return main_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libindelope_cuda has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from indelope_b200 import abi, api, cuda, host

    mode = scaling_mode(args)
    if mode == "strong" and WGS_CONTIGS % world:
        raise SystemExit("strong scaling deals %d contigs to the ranks in equal blocks: --gpus must divide it" % WGS_CONTIGS)
    cfg, ds, rois = build_workload(args.workload, rank, world, args.scale, mode)
    n_regions, n_reads = rois.n_rois, rois.total_reads()
    caller = api.Caller(local, **CALL)
    ctx, P = caller.ctx, caller.params

    def alloc_pack(lo, hi):
        nr, sb, rb = rois.pack_size(lo, hi, P)
        b = ctx.batch_alloc(hi - lo + 1, nr + 1, sb + 64, rb + 64)
        rois.pack(lo, hi, P, b)
        return b, (hi - lo) * C.sizeof(abi.Region) + nr * C.sizeof(abi.Read) + sb // 4 + sb // 8 + rb // 4 + rb // 8

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def result_bytes(r):
        return (r.n_regions * C.sizeof(abi.RegionResult) + r.n_contigs * C.sizeof(abi.ContigResult) + r.n_alns * C.sizeof(abi.AlnResult) +
                r.n_events * C.sizeof(abi.EventResult) + r.n_cigar_ops * 4 + r.n_contig_bases)

    sampler = ClockSampler(local)
    extra, dumped = {}, {}
    if mode == "weak":
        # ---- pinned batches: one big batch for the device-resident leg, `e2e_batches` slices for the end-to-end legs
        big, big_bytes = alloc_pack(0, n_regions)
        cuts = [n_regions * i // args.e2e_batches for i in range(args.e2e_batches + 1)]
        spans = [(cuts[i], cuts[i + 1]) for i in range(args.e2e_batches) if cuts[i + 1] > cuts[i]]
        slices = [alloc_pack(a, b) for a, b in spans]
        # ---- leg 1: inputs resident in HBM, kernels only (CUDA events on the library's stream)
        ctx.upload(big)

        def resident_step():
            t = ctx.run_resident(big)
            r = ctx.wait(t).contents
            d = {k: getattr(r, k) for k in KEYS}
            ctx.release(t)
            return d
        for _ in range(args.warmup):
            resident_step()
        sampler.start()
        barrier()
        steps = [resident_step() for _ in range(args.steps)]
        barrier()
        dev_ms = sum(s["ms_total"] for s in steps)
        launches = sum(s["kernel_launches"] for s in steps)

        # ---- leg 2: end to end through the C ABI with HOST (pinned) buffers: H2D + kernels + D2H of every result.  The caller streams
        # batches as the reference-facing API intends (idl_submit / idl_wait with tickets, `n_streams` batches in flight): the pipeline
        # runs on across step boundaries and is drained once, inside the timed region, before the closing barrier.  repack=True also
        # re-packs every batch from the ASCII reads on the host cores (idlh_pack: quality trim, 2-bit packing, records) each step.
        def e2e_steps(k, repack, held=None):
            inflight, d2h, nl, kern = [], 0, 0, 0.0

            def retire():
                nonlocal d2h, nl, kern
                t, last = inflight.pop(0); r = ctx.wait(t).contents; d2h += result_bytes(r); nl += r.kernel_launches
                kern += sum(getattr(r, s) for s in STAGES)
                if last:   # --dump-outputs: the last step's tickets stay unreleased, in batch order, until the timed window has closed
                    held.append((t, r))
                else:
                    ctx.release(t)
            for s in range(k):
                for (b, _), (lo, hi) in zip(slices, spans):
                    if len(inflight) >= P.n_streams:
                        retire()
                    if repack:
                        rois.pack(lo, hi, P, b)
                    inflight.append((ctx.submit(b), held is not None and s == k - 1))
            while inflight:
                retire()
            return d2h, nl, kern

        def timed_e2e(repack, held=None):
            e2e_steps(args.warmup, repack)
            barrier()
            t0 = time.perf_counter()
            d2h, nl, kern = e2e_steps(args.steps, repack, held)
            barrier()
            return time.perf_counter() - t0, d2h // max(1, args.steps), nl, kern
        if args.dump_outputs and len(slices) > P.n_streams:
            # a held ticket keeps its lane: the last step's batches must all be in flight at once
            raise SystemExit("--dump-outputs needs --e2e-batches <= %d (the library's streams)" % P.n_streams)
        held = [] if args.dump_outputs else None
        e2e_s, d2h_bytes, nl, e2e_kern_ms = timed_e2e(False, held)
        if args.dump_outputs:
            dumped = dump_results([result_tables(r) for _, r in held])
            for t, _ in held:
                ctx.release(t)
        launches += nl
        pk_s, _, nl, pk_kern_ms = timed_e2e(True)
        launches += nl
        h2d_bytes = sum(b for _, b in slices)
        extra["e2e_packed_ms"] = pk_s * 1000.0
        tp0 = time.perf_counter()
        for (b, _), (lo, hi) in zip(slices, spans):
            rois.pack(lo, hi, P, b)
        extra["pack_ms"] = (time.perf_counter() - tp0) * 1000.0
        merged = None
        # ---- leg 4 (N=1): the same regions from a BAM RESIDENT ON THE DEVICE: the workload written as a BAM file, decoded by idl_bam_open (inflate, record
        # chaining, fields), every batch BUILT ON THE DEVICE by idl_bam_submit (quality trim, windows, records, 2-bit pools from the BAM's nibbles) and run;
        # per step only the regions' coordinates and record indices go up, the results come down.  Compare with e2e_packed, where the host packs.
        if world == 1 and not args.no_bam_leg:
            try:
                import shutil
                import tempfile
                tmpd = tempfile.mkdtemp(prefix="idl_bench_")
                try:
                    bam_path = os.path.join(tmpd, "w.bam")
                    tw = time.perf_counter(); ds.write_bam(bam_path, level=1); write_s = time.perf_counter() - tw
                    data = open(bam_path, "rb").read()
                finally:
                    shutil.rmtree(tmpd, ignore_errors=True)
                cuda.Bam(data, device=local).close()   # first use: module load, allocator warm-up
                to = time.perf_counter(); bamdev = cuda.Bam(data, device=local); open_s = time.perf_counter() - to
                arr = rois.arrays()
                for c in range(bamdev.n_ref):
                    bamdev.set_reference(c, arr["chrom_seqs"][c])
                rbeg = np.concatenate([arr["roi_read_begin"], [len(arr["read_idx"])]]).astype(np.int64)
                bam_slices = [(np.ascontiguousarray(arr["roi_chrom"][lo:hi]), np.ascontiguousarray(arr["roi_start"][lo:hi]), np.ascontiguousarray(arr["roi_stop"][lo:hi]),
                               np.ascontiguousarray(arr["roi_n_reads"][lo:hi]), np.ascontiguousarray(arr["read_idx"][rbeg[lo]:rbeg[hi]]), lo) for lo, hi in spans]

                def bam_steps(k):
                    inflight, nl, kern, sig = [], 0, 0.0, []

                    def retire():
                        nonlocal nl, kern
                        t = inflight.pop(0); r = ctx.wait(t).contents; nl += r.kernel_launches + 9
                        kern += sum(getattr(r, s) for s in STAGES); sig.append((r.n_regions, r.n_contigs, r.n_alns, r.n_events, r.n_cigar_ops)); ctx.release(t)
                    for _ in range(k):
                        for ch, st_, en, nr_, idx, lo in bam_slices:
                            if len(inflight) >= P.n_streams:
                                retire()
                            inflight.append(ctx.bam_submit(bamdev, ch, st_, en, nr_, idx, ordinal_base=lo))
                    while inflight:
                        retire()
                    return nl, kern, sig
                _, _, sig_bam = bam_steps(max(1, args.warmup))
                # the same work as the host-packed batches: result counts of every batch agree
                ref_sig = []
                for (b, _), _ in zip(slices, spans):
                    t = ctx.submit(b); r = ctx.wait(t).contents; ref_sig.append((r.n_regions, r.n_contigs, r.n_alns, r.n_events, r.n_cigar_ops)); ctx.release(t)
                bam_ok = sig_bam[:len(ref_sig)] == ref_sig
                kb = max(1, args.steps // 2)
                barrier()
                t0 = time.perf_counter()
                nl, bam_kern, _ = bam_steps(kb)
                barrier()
                bam_s = time.perf_counter() - t0
                launches += nl
                extra["e2e_bam"] = {"value": n_regions * kb / bam_s, "unit": "regions/s", "steps": kb, "ms_per_step": bam_s * 1000.0 / kb, "kernel_ms_per_step": bam_kern / kb,
                                    "h2d_bytes_per_step": int(n_regions * 16 + len(arr["read_idx"]) * 8), "same_result_counts_as_host_packed_batches": bool(bam_ok),
                                    "bam": {"file_bytes": len(data), "write_s": write_s, "idl_bam_open_wall_s": open_s, **bamdev.info, "records": bamdev.n_records},
                                    "what": "regions from a BAM resident on the device: idl_bam_open once (outside the timed region), then per step every batch is built on the device "
                                            "by idl_bam_submit (quality trim, windows, records, 2-bit pools from the BAM's nibbles) and run; results copied back as in e2e"}
                bamdev.close()
            except Exception as ex:   # this leg is an extra: it must never cost the run its bench line
                extra["e2e_bam"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    else:
        # ---- strong scaling: this rank's block of contigs in pinned batches; per step every batch goes through submit / wait / the host
        # cascade (filters, genotype likelihoods, VCF text), then the shards' records are gathered on rank 0 and deduped
        plans = api.plan_batches(rois, 0, n_regions, max_reads=1_200_000, max_regions=60_000)
        slices = [alloc_pack(a, b) for a, b in plans]
        big_bytes = sum(b for _, b in slices)
        writer_params = P

        bufs = {}

        def strong_step(collect):
            inflight, texts, d2h, nl, stats, host_s = [], [], 0, 0, [], 0.0
            writer = host.VcfWriter(dedup=False)

            def retire():
                nonlocal d2h, nl, host_s
                (a, b), t = inflight.pop(0)
                res = ctx.wait(t); r = res.contents
                d2h += result_bytes(r); nl += r.kernel_launches
                stats.append({k: getattr(r, k) for k in KEYS})
                th = time.perf_counter()
                v = writer.records_bytes(rois, a, writer_params, res)
                host_s += time.perf_counter() - th
                ctx.release(t)
                texts.append(v)
            for (b, _), span in zip(slices, plans):
                if len(inflight) >= P.n_streams:
                    retire()
                inflight.append((span, ctx.submit(b)))
            while inflight:
                retire()
            mine = b"".join(texts)
            tm = time.perf_counter()
            # the only communication of the run: the shards' record text (bytes) to rank 0 over NCCL, into buffers that are reused from step
            # to step (fresh 60 MB allocations cost more in page faults than the merge itself), then the dedup in place
            n_mine = len(mine)
            if world > 1:
                ln = torch.tensor([n_mine], dtype=torch.int64, device="cuda")
                lens = [torch.zeros_like(ln) for _ in range(world)]
                dist.all_gather(lens, ln)
                lens = [int(x.item()) for x in lens]
                cap = (max(lens) + 1023) // 1024 * 1024
                if bufs.get("cap", 0) < cap:
                    bufs["cap"] = cap
                    bufs["send"] = torch.zeros(cap, dtype=torch.uint8, device="cuda")
                    bufs["stage"] = torch.empty(cap, dtype=torch.uint8).pin_memory()
                    bufs["parts"] = [torch.empty(cap, dtype=torch.uint8, device="cuda") for _ in range(world)] if rank == 0 else None
                cap = bufs["cap"]
                if n_mine:
                    bufs["stage"][:n_mine] = torch.frombuffer(mine, dtype=torch.uint8)
                    bufs["send"][:n_mine].copy_(bufs["stage"][:n_mine], non_blocking=True)
                dist.gather(bufs["send"], bufs["parts"], dst=0)
                total = sum(lens)
            else:
                total = n_mine
            out = None
            if rank == 0:
                if bufs.get("hcap", 0) < total + 1:
                    bufs["hcap"] = total + 1 + (total >> 3)
                    bufs["host"] = torch.empty(bufs["hcap"], dtype=torch.uint8).pin_memory()
                hbuf = bufs["host"]
                if world > 1:
                    at = 0
                    for p, n in zip(bufs["parts"], lens):
                        hbuf[at:at + n].copy_(p[:n], non_blocking=True); at += n
                    torch.cuda.synchronize()
                elif total:
                    hbuf[:total] = torch.frombuffer(mine, dtype=torch.uint8)
                kept = host.dedup_inplace(hbuf.data_ptr(), total)
                if collect:
                    out = bytes(hbuf[:kept].numpy().data)
            merge_s = time.perf_counter() - tm
            return d2h, nl, stats, host_s, merge_s, (out if collect else None), (mine if collect else None)
        for _ in range(args.warmup):
            strong_step(False)
        sampler.start()
        barrier()
        t0 = time.perf_counter()
        acc = [strong_step(False) for _ in range(max(0, args.steps - 1))] + [strong_step(True)]
        barrier()
        e2e_s = time.perf_counter() - t0
        d2h_bytes = sum(a[0] for a in acc) // max(1, args.steps)
        launches = sum(a[1] for a in acc)
        steps = [{k: sum(b[k] for b in a[2]) for k in KEYS} for a in acc]  # per step: summed over the batches
        dev_ms = sum(sum(s[k] for k in STAGES) for s in steps)             # device kernel time (CUDA events around each stage of each batch), copies excluded
        e2e_kern_ms = dev_ms
        h2d_bytes = big_bytes
        extra["host_cascade_ms_per_step"] = 1000.0 * sum(a[3] for a in acc) / args.steps
        extra["merge_ms_per_step"] = 1000.0 * sum(a[4] for a in acc) / args.steps
        merged, mine_raw = acc[-1][5], acc[-1][6]
        if rank == 0 and args.dump_outputs:
            dumped = dump_text(merged)
    sampler.stop_flag = True; sampler.join(timeout=2)

    # max over ranks
    tt = torch.tensor([dev_ms, e2e_s * 1000.0, extra.get("e2e_packed_ms", 0.0)], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(n_regions), float(n_reads), float(h2d_bytes), float(d2h_bytes)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_ms_max, pk_ms_max = tt.tolist(); regions_all, reads_all, h2d_all, d2h_all = tot.tolist()  # whole job: summed over ranks

    verify = None
    if mode == "strong" and args.verify:
        # the checker: every rank runs the CPU oracle on its own block (raw records), rank 0 merges them with its own restatement of the dedup
        _, _, ocnt, use_ref, oraw = run_oracle(rois, rois.n_rois, os.cpu_count() or 1, raw=True)
        if world > 1:
            og = [None] * world if rank == 0 else None
            dist.gather_object(oraw, og, dst=0)
        else:
            og = [oraw]
        if rank == 0:
            want = dedup_text("".join(og))
            merged = merged.decode()
            verify = {"merged_vcf_equals_oracle": merged == want, "records": merged.count("\n"), "oracle_records": want.count("\n"),
                      "oracle_dp": "reference ksw2_extz2_sse.c (oracle/_ref)" if use_ref else "lane model"}

    if rank == 0:
        K = args.steps
        avg = {k: sum(s[k] for s in steps) / K for k in KEYS}
        value = regions_all * K / (dev_ms_max / 1000.0)
        e2e_val = regions_all * K / (e2e_ms_max / 1000.0)
        peak, peak_src, sm_max = load_peaks()
        # the kernel that serves call-site A under the current settings (pipeline.cu launch_chain): four threads per alignment by default
        site_a = "align_band_kernel" if os.environ.get("IDL_BAND_REGS") == "1" else ("align_kernel" if os.environ.get("IDL_ALIGN_G") == "8" else "align4_kernel")
        kern = {"assemble_kernel": avg["ms_assemble"], site_a: avg["ms_align"], "kmer_kernel": avg["ms_genotype"], "al_kernel": avg["ms_al"]}
        dom = max(kern, key=kern.get)
        # algorithmic bytes per launch of each kernel (DESIGN.md "Kernels"): what the kernel must read + write once
        pk_bytes = big_bytes if mode == "weak" else h2d_bytes
        alg = {
            "assemble_kernel": pk_bytes + avg["n_contigs"] * 24 + n_regions * 16,
            site_a: avg["dp_cells_a"] * 1.0 + avg["n_alns"] * 72,   # one backtrack byte per in-band cell + the result record
            "kmer_kernel": avg["kmer_bytes"],
            "al_kernel": avg["dp_cells_b"] * 1.0,
        }
        hbm_gbs = alg[dom] / (kern[dom] / 1000.0) / 1e9 if kern[dom] > 0 else 0.0
        # DRAM bytes, executed thread instructions and ALU-pipe utilisation per launch of the dominant kernel come from the committed ncu
        # capture of this exact command (profiles/r02_traffic.json; default workload only): properties of the deterministic workload and of
        # the code, not of this run's timing -- a number taken under a profiler is never a bench value, so the timing here is live
        prof = {}
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath) and args.workload == "chr1" and args.scale == 1.0 and mode == "weak":
            prof = json.load(open(tpath)).get(dom, {})
        traffic = prof.get("dram_bytes_per_launch")
        clocks = sampler.summary()
        mhz = clocks.get("sm_mhz") or sm_max
        int_peak = 148 * 128 * mhz * 1e6 / 1e12  # Tiop/s: 128 INT32 lanes per SM x clock (the ALU and the FMA pipe together)
        ach = prof["thread_inst"] / (kern[dom] / 1000.0) / 1e12 if prof.get("thread_inst") and kern[dom] > 0 else None
        roofline = {
            "kernel": dom, "bound": "alu", "achieved": ach, "peak": int_peak, "unit": "Tiop/s", "frac": (ach / int_peak) if ach else None,
            "clock_mhz": mhz, "thread_inst_per_launch": prof.get("thread_inst"), "pipe_alu_busy_pct": prof.get("pipe_alu_pct"), "issue_active_pct": prof.get("issue_active_pct"),
            "traffic": traffic, "algorithmic_bytes": alg[dom], "traffic_ratio": (traffic / alg[dom]) if traffic and alg[dom] else None,
            "hbm_gbs": hbm_gbs, "hbm_peak_gbs": peak, "hbm_frac": hbm_gbs / peak, "dram_gbs": (traffic / (kern[dom] / 1000.0) / 1e9) if traffic and kern[dom] > 0 else None,
            "peak_source": "INT32 lanes x SM clock sampled under load; HBM: " + peak_src,
            "traffic_source": "profiles/r02_traffic.json (ncu capture of this command, launch 1: static per launch for a deterministic workload)" if prof else None,
            "note": "integer DP: the ALU pipe (IADD3/LOP3/SHF/PRMT/ISETP: one warp instruction per two cycles per scheduler) binds, `pipe_alu_busy_pct` is its "
                    "utilisation; `frac` counts every executed thread instruction against all 128 INT32 lanes per SM; the kernel must move one backtrack byte per DP cell (hbm_*)",
        }
        line = {
            "metric": "regions_per_s", "value": value, "unit": "regions/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / K, "higher_is_better": True, "scaling": mode, "vs_baseline": None, "dtype": "int8/int32/u64", "data": "synthetic",
            "reads_per_s": reads_all * K / (dev_ms_max / 1000.0),
            "ksw2_gcups": (avg["dp_cells_a"] + avg["dp_cells_b"]) / ((avg["ms_align"] + avg["ms_al"]) / 1000.0) / 1e9 if avg["ms_align"] + avg["ms_al"] > 0 else None,
            "ksw2_gcups_site_a": avg["dp_cells_a"] / (avg["ms_align"] / 1000.0) / 1e9 if avg["ms_align"] > 0 else None,
            "ksw2_gcups_site_b": avg["dp_cells_b"] / (avg["ms_al"] / 1000.0) / 1e9 if avg["ms_al"] > 0 else None,
            "kmer_gbs": avg["kmer_bytes"] / (avg["ms_genotype"] / 1000.0) / 1e9 if avg["ms_genotype"] > 0 else None,
            "assembler_offsets_per_s": avg["offsets_tested"] / (avg["ms_assemble"] / 1000.0) if avg["ms_assemble"] > 0 else None,
            "config": config_of(args, cfg, mode, rois),
            "run": {"l2": "inputs (%.0f MB packed per rank) exceed the 126 MB L2; no explicit flush" % (big_bytes / 1e6), "e2e_batches": len(slices), "streams": P.n_streams,
                    "e2e_pipelining": "batches streamed through idl_submit/idl_wait, %d in flight%s" % (
                        P.n_streams, ", across step boundaries, drained once inside the timed region" if mode == "weak" else "; every step ends with the gather and the dedup on rank 0"),
                    "value_clock": "CUDA events around the kernel chain, batch resident in HBM" if mode == "weak" else "sum of the CUDA-event stage times of every batch (copies excluded), max over ranks"},
            "kernel_ms": kern,
            "work": {k: avg[k] for k in ("offsets_tested", "dp_cells_a", "dp_cells_b", "dp_a", "dp_b", "kmer_reads", "kmer_bytes", "al_events", "n_contigs", "n_alns", "n_events")},
            "roofline": roofline,
            "e2e": {"value": e2e_val, "unit": "regions/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                    "ms_per_step": e2e_ms_max / K, "kernel_ms_per_step": e2e_kern_ms / K},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if mode == "weak":
            if "e2e_bam" in extra:
                line["e2e_bam"] = extra["e2e_bam"]
            line["e2e_packed"] = {"value": regions_all * K / (pk_ms_max / 1000.0), "unit": "regions/s", "ms_per_step": pk_ms_max / K, "pack_ms_per_step_alone": extra["pack_ms"],
                                  "pack_threads": min(32, os.cpu_count() or 1),
                                  "what": "as e2e, plus idlh_pack of every batch from the ASCII reads on the host cores inside the timed region (quality trim, 2-bit packing, read and region records)"}
        else:
            line["strong"] = {"contigs": WGS_CONTIGS, "contigs_per_rank": WGS_CONTIGS // world, "host_cascade_ms_per_step": extra["host_cascade_ms_per_step"],
                              "merge_ms_per_step": extra["merge_ms_per_step"], "merge_share_of_e2e": extra["merge_ms_per_step"] / (e2e_ms_max / K), "verify": verify}
        if world == 1:
            n, nr, cnt, use_ref, _ = run_oracle(rois, args.cpu_sample, 1)
            if cnt["offsets"] > 0 and avg["ms_assemble"] > 0:
                # SURVEY 8(d) secondary unit: exhaustive base compares (sum over tested offsets of the overlap length), the natural GPU
                # formulation -- ~100x the reference's early-abort count, never CPU-equivalent work.  The device counts offsets; the
                # compares per offset come from the oracle's counters on its sample of the same workload.
                line["assembler_exhaustive_compares_per_s"] = avg["offsets_tested"] * (cnt["exhaustive_compares"] / cnt["offsets"]) / (avg["ms_assemble"] / 1000.0)
                line["assembler_compares_per_offset"] = cnt["exhaustive_compares"] / cnt["offsets"]
            line["cpu_baseline"] = {"value": n / cnt["seconds"], "unit": "regions/s", "cores": 1, "kind": "port", "cpu": cpu_model(), "build": oracle_build_flags(),
                                    "reads_per_s": nr / cnt["seconds"], "seconds": cnt["seconds"],
                                    "ksw2_gcups": None if use_ref else (cnt["cells_a"] + cnt["cells_b"]) / cnt["seconds"] / 1e9,
                                    "sample": "first %d regions of the same workload, single thread (the reference is single-threaded on this path); CPU oracle%s" % (
                                        n, " calling the reference's own ksw2_extz2_sse.c compiled unmodified (oracle/_ref)" if use_ref else " with its own lane-exact ksw2")}
        if args.dump_outputs:
            write_dump(args.dump_outputs, dumped)
        print(json.dumps(line), file=OUT, flush=True)
    for b, _ in slices + ([(big, 0)] if mode == "weak" else []):
        ctx.batch_free(b)
    caller.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
