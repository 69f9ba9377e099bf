"""End-to-end timing of the `indelope` command line on real files (BAM -> VCF), next to its host-only share.
  python tools/cli_bench.py [chrom_len_mb] [threads] [qual_levels]      (qual_levels 8 or 40: per-base qualities, a BAM that compresses ~4:1 / ~3:1)
Writes a whole-contig 30x dataset (BASELINE config 1 scaled up: 200 planted indels per Mb) as .fa/.bam under a temp
directory, then times (1) the streaming sweep alone (BGZF inflate + BAM parse + gen_roi, no GPU), (2) the binary end to
end, and checks the binary's VCF against the CPU oracle run over the same regions (timed as the CPU baseline).
"""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from indelope_b200 import build, host


def main():
    mb = float(sys.argv[1]) if len(sys.argv) > 1 else 20.0
    threads = int(sys.argv[2]) if len(sys.argv) > 2 else 4
    levels = int(sys.argv[3]) if len(sys.argv) > 3 and sys.argv[3].isdigit() else 0
    cfg = dict(host.CONFIGS["pr1"]); cfg.update(chrom_len=int(mb * 1e6), n_events=int(200 * mb), qual_levels=levels)
    t0 = time.time(); ds = host.Dataset(**cfg); t_gen = time.time() - t0
    d = tempfile.mkdtemp(prefix="idl_cli_")
    fa, bam = os.path.join(d, "ref.fa"), os.path.join(d, "reads.bam")
    t0 = time.time(); ds.write_fasta(fa); ds.write_bam(bam, level=1); t_write = time.time() - t0
    out = {"chrom_len": cfg["chrom_len"], "qual_levels": levels, "reads": ds.n_reads, "bam_bytes": os.path.getsize(bam), "threads": threads, "gen_s": round(t_gen, 2), "write_s": round(t_write, 2)}
    t0 = time.time()
    st = host.Stream(fa, bam, threads=threads, min_reads=5)
    groups = list(st.groups())
    out["host_sweep_s"] = round(time.time() - t0, 3)
    out["regions"] = sum(g.n_rois for g in groups); out["region_reads"] = sum(g.total_reads() for g in groups)
    exe = build.build_cli()
    if "--host-only" not in sys.argv:
        best = None
        for _ in range(3):
            t0 = time.time()
            r = subprocess.run([exe, "--min-event-len", "5", "--min-reads", "5", "-t", str(threads), fa, bam], capture_output=True, text=True,
                               env=dict(os.environ, INDELOPE_TIMING="1"))
            dt = time.time() - t0
            if r.returncode != 0:
                out["cli_error"] = r.stderr[-300:]; break
            if best is None or dt < best:
                best = dt; out["cli_phases"] = r.stderr.strip().split("\n")[-1]
        if best is not None:
            out["cli_s"] = round(best, 3); out["cli_reads_per_s"] = round(ds.n_reads / best); out["cli_regions_per_s"] = round(out["regions"] / best)
            out["vcf_records"] = sum(1 for l in r.stdout.split("\n") if l and not l.startswith("#"))
            from oracle import pyoracle as orc
            t0 = time.time(); vcf = ""
            for g in groups:
                pass
            whole = ds.sweep(min_reads=5)
            _, ovcf, cnt = orc.call(whole.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=0, n_threads=os.cpu_count() or 1)
            out["oracle_s_all_threads"] = round(time.time() - t0, 3); out["oracle_threads"] = os.cpu_count()
            out["vcf_identical_to_oracle"] = (r.stdout == whole.header() + ovcf)
            # the same command with the front end on the GPU (idl_bam_open / idl_bam_sweep / idl_bam_submit)
            best = None
            for _ in range(3):
                t0 = time.time()
                r2 = subprocess.run([exe, "--gpu-decode", "--min-event-len", "5", "--min-reads", "5", fa, bam], capture_output=True, text=True,
                                    env=dict(os.environ, INDELOPE_TIMING="1", IDL_BAM_TIMING="1"))
                dt = time.time() - t0
                if r2.returncode != 0:
                    out["gpu_decode_error"] = r2.stderr[-300:]; break
                if best is None or dt < best:
                    best = dt; out["gpu_decode_phases"] = r2.stderr.strip().split("\n")[-2:]
            if best is not None:
                out["gpu_decode_cli_s"] = round(best, 3); out["gpu_decode_vcf_identical_to_oracle"] = (r2.stdout == whole.header() + ovcf)
            # ... and target by target through the index, as the binary decodes a file larger than an eighth of the free device memory
            r3 = subprocess.run([exe, "--gpu-decode", "--min-event-len", "5", "--min-reads", "5", fa, bam], capture_output=True, text=True,
                                env=dict(os.environ, INDELOPE_TIMING="1", INDELOPE_BY_TARGET="1"))
            if r3.returncode == 0:
                out["gpu_decode_by_target_phases"] = r3.stderr.strip().split("\n")[-1]; out["gpu_decode_by_target_vcf_identical_to_oracle"] = (r3.stdout == whole.header() + ovcf)
            else:
                out["gpu_decode_by_target_error"] = r3.stderr[-300:]
            # the decoders alone, in process: host reader (inflate + parse on `threads` host threads) against idl_bam_open
            from indelope_b200 import cuda
            data = open(bam, "rb").read()
            t0 = time.time(); full = host.Dataset.load(fa, bam, threads=threads); out["host_load_s"] = round(time.time() - t0, 3)
            del full
            cuda.Bam(data).close()  # context + first-touch
            best = None
            for _ in range(3):
                t0 = time.time(); b = cuda.Bam(data); dt = time.time() - t0
                if best is None or dt < best:
                    best = dt; out["idl_bam_open"] = dict(b.info, wall_s=round(dt, 4), n_records=b.n_records)
                b.close()
            i = out["idl_bam_open"]
            out["copy_inflate_gbs_out"] = round(i["inflated_bytes"] / (i["ms_inflate"] / 1e3) / 1e9, 2)
            out["idl_bam_open_gbs_out"] = round(i["inflated_bytes"] / i["wall_s"] / 1e9, 2)
    print(json.dumps(out))
    for f in (fa, fa + ".fai", bam, bam + ".bai"):
        if os.path.exists(f):
            os.remove(f)
    os.rmdir(d)


if __name__ == "__main__":
    main()
