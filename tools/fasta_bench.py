"""A bgzipped reference on the GPU (idl_fasta_open) next to the host loaders, on a genome-size synthetic reference.
  python tools/fasta_bench.py [--chroms N] [--mb MB_PER_CHROM] [--no-cli]
The reference of `--workload wgs` (24 x 129 Mb by default): the generator's sequence with soft-masked stretches and N runs, written plain in 60 columns,
bgzipped (BGZF members of 0xff00 bytes, deflate level 6), and as an unwrapped variant (one line per record).  Building the files is not timed.
Times: the host loader on the plain file and on the .fa.gz with 1 and with all threads; idl_fasta_open by phase (reading the file, H2D, inflate, parse,
copy-back of every sequence); the parse's rate of algorithmic and of streamed bytes next to the HBM copy rate measured in the same run; and the wall
time of `indelope -g` and of a one-interval `indelope -r` over a BAM with a few thousand reads, with the .fa and with the .fa.gz.
"""
import json
import multiprocessing as mp
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from indelope_b200 import build, cuda, host  # noqa: E402


def _member(chunk):
    import struct
    co = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
    c = co.compress(chunk) + co.flush()
    return b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", 18 + len(c) + 8 - 1) + c + struct.pack("<II", zlib.crc32(chunk), len(chunk))


def bgzip(src, dst):
    data = open(src, "rb").read()
    with mp.Pool() as pool, open(dst, "wb") as f:
        for m in pool.imap(_member, (data[i:i + 0xff00] for i in range(0, len(data), 0xff00)), chunksize=64):
            f.write(m)
        f.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))


def write_fasta(path, names, seqs, width):
    with open(path, "wb") as f:
        for n, s in zip(names, seqs):
            f.write(b">" + n.encode() + b" synthetic\n")
            if width:
                pad = (-len(s)) % width
                a = np.concatenate([s, np.full(pad, 10, np.uint8)]).reshape(-1, width)
                lines = np.concatenate([a, np.full((len(a), 1), 10, np.uint8)], axis=1).ravel()
                f.write(lines[:len(lines) - pad].tobytes() if pad else lines.tobytes())
            else:
                f.write(s.tobytes() + b"\n")


def timed(f):
    t0 = time.time(); r = f(); return r, round(time.time() - t0, 3)


def device_open(path):
    t0 = time.time(); data = open(path, "rb").read(); t_read = time.time() - t0
    t0 = time.time(); fa = cuda.Fasta(data); t_open = time.time() - t0
    t0 = time.time(); seqs = [fa.sequence(r) for r in range(fa.n_records)]; t_back = time.time() - t0
    i = fa.info
    out = dict(read_s=round(t_read, 3), open_wall_s=round(t_open, 3), ms_h2d=round(i["ms_h2d"], 2), ms_inflate=round(i["ms_inflate"], 2), ms_parse=round(i["ms_parse"], 2),
               copy_back_s=round(t_back, 3), file_bytes=i["file_bytes"], inflated_bytes=i["inflated_bytes"], sequence_bytes=i["sequence_bytes"], n_members=i["n_members"],
               parse_gbs_algorithmic=round(i["parse_algorithmic_bytes"] / i["ms_parse"] / 1e6, 1), parse_gbs_streamed=round(i["parse_streamed_bytes"] / i["ms_parse"] / 1e6, 1),
               inflate_gbs_out=round(i["inflated_bytes"] / i["ms_inflate"] / 1e6, 1))
    fa.close()
    return out, seqs


def hbm_copy_gbs():
    import torch
    x = torch.empty(4 << 30, dtype=torch.uint8, device="cuda"); y = torch.empty_like(x)
    for _ in range(3):
        y.copy_(x)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        y.copy_(x)
    b.record(); torch.cuda.synchronize()
    gbs = 10 * 2 * x.numel() / (a.elapsed_time(b) / 1e3) / 1e9   # read + write
    del x, y
    torch.cuda.empty_cache()
    return round(gbs, 1)


def main():
    argv = sys.argv[1:]
    opt = lambda k, d: type(d)(argv[argv.index(k) + 1]) if k in argv else d  # noqa: E731
    n_chroms, mb = opt("--chroms", 24), opt("--mb", 129.0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True) if shutil.which("nvidia-smi") else None
    out = {"gpu": smi.stdout.strip() if smi else "no nvidia-smi"}
    d = tempfile.mkdtemp(prefix="idl_fasta_")
    try:
        cfg = dict(host.CONFIGS["wgs"]); cfg.update(n_chroms=n_chroms, chrom_len=int(mb * 1e6), n_events=4)
        ds = host.Dataset(**cfg)
        names, seqs = ds.sequences()
        rng = np.random.default_rng(1)
        masked = []
        for s in seqs:
            s = np.array(s, dtype=np.uint8)
            for _ in range(max(1, len(s) // 200_000)):   # soft-masked repeats and N runs
                a = int(rng.integers(0, len(s) - 5000)); k = int(rng.integers(100, 5000))
                s[a:a + k] = s[a:a + k] | 0x20 if rng.random() < 0.8 else ord("N")
            masked.append(s)
        fa, gz, un, ungz, bam = (os.path.join(d, x) for x in ("ref.fa", "ref.fa.gz", "unwrapped.fa", "unwrapped.fa.gz", "reads.bam"))
        write_fasta(fa, names, masked, 60); write_fasta(un, names, masked, 0)
        bgzip(fa, gz); bgzip(un, ungz)
        ds.write_bam(bam, level=6)
        out.update(genome_bases=int(sum(len(s) for s in masked)), fa_bytes=os.path.getsize(fa), fa_gz_bytes=os.path.getsize(gz), reads=ds.n_reads)
        del ds, seqs
        want = [bytes(s) for s in masked]; del masked
        _, out["host_plain_s"] = timed(lambda: host.Dataset.load_fasta(fa))
        for th in (1, os.cpu_count() or 1):
            host.set_threads(th)
            _, out["host_bgzf_s_%dthr" % th] = timed(lambda: host.Dataset.load_fasta(gz))
        host.set_threads(0)
        out["hbm_copy_gbs"] = hbm_copy_gbs()
        device_open(gz)   # warm-up: context, module load
        for label, path in (("device_wrapped", gz), ("device_unwrapped", ungz)):
            best = None
            for _ in range(3):
                r, got = device_open(path)
                if best is None or r["open_wall_s"] < best["open_wall_s"]:
                    best = r
            assert [bytes(x) for x in got] == want, label
            best["parse_share_of_copy"] = round(best["parse_gbs_streamed"] / out["hbm_copy_gbs"], 2)
            out[label] = best
        if "--no-cli" not in argv:
            exe = build.build_cli()
            for label, args in (("cli_g", ["-g"]), ("cli_r", ["-r", "%s:1000000-1100000" % names[0]])):
                res = {}
                for ref in (fa, gz, fa, gz):
                    t0 = time.time()
                    r = subprocess.run([exe] + args + [ref, bam], capture_output=True)
                    dt = round(time.time() - t0, 3)
                    assert r.returncode == 0, r.stderr.decode()[-2000:]
                    key = "fa_gz" if ref == gz else "fa"
                    res.setdefault(key + "_s", []).append(dt)
                    res[key + "_stdout"] = r.stdout
                assert res["fa_stdout"] == res["fa_gz_stdout"], label
                out[label] = {k: v for k, v in res.items() if not k.endswith("stdout")}
    finally:   # what was measured so far, also when interrupted
        print(json.dumps(out), flush=True)
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
