"""Wall time of `indelope -R targets.bed` against the whole-file `indelope --gpu-decode` run on the tools/cli_bench.py BAM.
  python tools/region_bench.py [chrom_len_mb] [reps]
Writes the whole-contig 30x dataset of tools/cli_bench.py (200 planted indels per Mb) as .fa/.bam under a temp directory, then times the binary with BEDs of
1, 100 and 10 000 random intervals (seeded) and without any, best of `reps`.  For each it reports wall time, the bytes read and decoded, slices, retries and
regions from INDELOPE_TIMING, and whether the VCF equals the CPU oracle's over the whole-file regions that overlap the intervals.  Prints one JSON line; the
card's name and power limit are read in the same run.
"""
import json
import os
import random
import re
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from indelope_b200 import build, host  # noqa: E402
from oracle import pyoracle as orc  # noqa: E402


def timed(exe, args, reps):
    best, r = None, None
    for _ in range(reps):
        t0 = time.time()
        r = subprocess.run([exe, "--min-event-len", "5", "--min-reads", "5"] + args, capture_output=True, text=True, env=dict(os.environ, INDELOPE_TIMING="1"))
        dt = time.time() - t0
        if r.returncode != 0:
            raise SystemExit("indelope failed: " + r.stderr[-500:])
        if best is None or dt < best[0]:
            best = (dt, r)
    return best


def main():
    mb = float(sys.argv[1]) if len(sys.argv) > 1 else 20.0
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    cfg = dict(host.CONFIGS["pr1"]); cfg.update(chrom_len=int(mb * 1e6), n_events=int(200 * mb))
    ds = host.Dataset(**cfg)
    d = tempfile.mkdtemp(prefix="idl_region_")
    try:
        fa, bam = os.path.join(d, "ref.fa"), os.path.join(d, "reads.bam")
        ds.write_fasta(fa); ds.write_bam(bam, level=1)
        name = ds.sequences()[0][0]
        L = cfg["chrom_len"]
        out = {"chrom_len": L, "bam_bytes": os.path.getsize(bam), "reads": ds.n_reads}
        try:
            out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
        except OSError:
            out["gpu"] = "unknown"
        whole = ds.sweep(min_reads=5)
        arrays = whole.arrays()
        rs, re_ = np.asarray(arrays["roi_start"]), np.asarray(arrays["roi_stop"])
        exe = build.build_cli()
        dt, r = timed(exe, ["--gpu-decode", fa, bam], reps)
        out["whole_file_gpu_decode_s"] = round(dt, 3)
        rng = random.Random(2026)
        out["beds"] = []
        for n in (1, 100, 10_000):
            ivs = sorted((b, min(L, b + rng.choice([200, 1000, 5000]))) for b in (rng.randrange(0, L) for _ in range(n)))
            bed = os.path.join(d, "t%d.bed" % n)
            with open(bed, "w") as f:
                f.writelines("%s\t%d\t%d\n" % (name, b, e) for b, e in ivs)
            dt, r = timed(exe, ["-R", bed, fa, bam], reps)
            line = [l for l in r.stderr.splitlines() if l.startswith("indelope timing (regions)")][-1]
            pats = dict(read=r"([\d.]+) MB read", decoded=r"([\d.]+) MB decoded", slices=r"slices (\d+)", retries=r"retries (\d+)", regions=r"regions (\d+)")
            nums = {k: float(re.search(p, line).group(1)) for k, p in pats.items()}
            b_arr = np.array([x[0] for x in ivs]); e_arr = np.array([x[1] for x in ivs])
            j = np.searchsorted(b_arr, re_, side="right")        # intervals starting at or before roi_end; overlap iff one of them ends after roi_start
            emax = np.maximum.accumulate(e_arr)
            keep = [k for k in range(len(rs)) if j[k] > 0 and emax[j[k] - 1] > rs[k]]
            ovcf = orc.call(util_subset(arrays, keep), min_reads=5, min_ctg_len=73, min_event_len=5, dump_level=0, n_threads=os.cpu_count() or 1)[1] if keep else ""
            out["beds"].append(dict(intervals=n, wall_s=round(dt, 3), mb_read=nums.get("read"), mb_decoded=nums.get("decoded"), slices=int(nums.get("slices", -1)),
                                    retries=int(nums.get("retries", -1)), regions=int(nums.get("regions", -1)), vcf_identical_to_oracle=r.stdout == whole.header() + ovcf))
        print(json.dumps(out))
    finally:
        shutil.rmtree(d, ignore_errors=True)


def util_subset(arrays, keep):
    """the same reads with only the regions in `keep` (tests/idl_testutil.py region_subset)"""
    keep = np.asarray(sorted(keep), np.int64)
    out = dict(arrays)
    for k in ("roi_chrom", "roi_start", "roi_stop", "roi_read_begin", "roi_n_reads"):
        out[k] = np.asarray(arrays[k])[keep]
    return out


if __name__ == "__main__":
    main()
