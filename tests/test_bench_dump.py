"""bench.py --dump-outputs: the result tables of a step come out in the order a caller reads them, whatever order the device handed
out its slots in and however the step was cut into batches, within 64 MB; on the device, two runs with the same arguments write the
same arrays."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from indelope_b200 import abi

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# regions -> contigs -> alignment (or none) -> CIGAR ops and event records
REGIONS = [
    dict(status=0, pre=3, contigs=[dict(start=100, nreads=7, seq=b"ACGTA", aln=dict(score=5, cigar=[0x50, 0x21, 0x30], events=[(1 << 50) + 7, 12])),
                                   dict(start=140, nreads=4, seq=b"GGC", aln=None)]),
    dict(status=2, pre=0, contigs=[]),
    dict(status=0, pre=2, contigs=[dict(start=300, nreads=9, seq=b"TTAC", aln=dict(score=-3, cigar=[0x40], events=[])),
                                   dict(start=333, nreads=5, seq=b"CAGGTT", aln=dict(score=1, cigar=[0x12, 0x31], events=[99]))]),
]


class Pool:
    """slots handed out front to back, or back to front (as a device may, in completion order)"""

    def __init__(self, total, rev):
        self.total, self.rev, self.used = total, rev, 0

    def take(self, n):
        at = self.used; self.used += n
        return self.total - at - n if self.rev else at


def results(rev, regions=REGIONS):
    ctgs = [c for r in regions for c in r["contigs"]]
    alns = [c["aln"] for c in ctgs if c["aln"]]
    reg = (abi.RegionResult * len(regions))(); ctg = (abi.ContigResult * len(ctgs))(); aln = (abi.AlnResult * len(alns))()
    ev = (abi.EventResult * sum(len(a["events"]) for a in alns))(); cig = (C.c_uint32 * sum(len(a["cigar"]) for a in alns))()
    seq = C.create_string_buffer(sum(len(c["seq"]) for c in ctgs))
    pc, pa, pe, po, ps = (Pool(len(x), rev) for x in (ctg, aln, ev, cig, seq.raw))
    for ri, r in enumerate(regions):
        cb = pc.take(len(r["contigs"]))
        reg[ri].status, reg[ri].n_contigs_pre, reg[ri].n_contigs, reg[ri].contig_begin = r["status"], r["pre"], len(r["contigs"]), cb
        for k, c in enumerate(r["contigs"]):
            o = ctg[cb + k]
            o.start, o.nreads, o.len, o.region, o.seq_off, o.aln = c["start"], c["nreads"], len(c["seq"]), ri, ps.take(len(c["seq"])), -1
            seq[o.seq_off:o.seq_off + o.len] = c["seq"]
            if c["aln"]:
                a = c["aln"]; ai = pa.take(1); o.aln = ai; x = aln[ai]
                x.region, x.contig, x.score, x.n_cigar, x.cigar_off, x.n_events = ri, cb + k, a["score"], len(a["cigar"]), po.take(len(a["cigar"])), len(a["events"])
                x.event_begin = pe.take(len(a["events"])) if a["events"] else bench.NO_EVENTS
                for j, op in enumerate(a["cigar"]):
                    cig[x.cigar_off + j] = op
                for j, code in enumerate(a["events"]):
                    e = ev[x.event_begin + j]; e.aln, e.index, e.ref_code = ai, j, code
    r = abi.Results(n_regions=len(reg), n_contigs=len(ctg), n_alns=len(aln), n_events=len(ev), n_cigar_ops=len(cig), n_contig_bases=len(seq.raw))
    r.region, r.contig, r.aln, r.event = reg, ctg, aln, ev
    r.cigar, r.contig_seq = cig, C.cast(seq, C.POINTER(C.c_char))
    return bench.result_tables(r)


def test_dump_is_independent_of_the_slot_order_and_the_batches():
    a, b = results(False), results(True)
    assert a["ctg"]["start"][0] != b["ctg"]["start"][0]          # the two layouts differ
    da, db = bench.dump_results([a]), bench.dump_results([b])
    dc = bench.dump_results([results(True, REGIONS[:1]), results(False, REGIONS[1:])])   # the same step in two batches
    assert sorted(da) == sorted(db) == ["alignments", "cigar", "contig_bases", "contigs", "counts", "events", "regions"]
    for k in da:
        assert np.array_equal(da[k], db[k]) and np.array_equal(da[k], dc[k]), k
        assert da[k].dtype in (np.float32, np.float64), k
    assert da["regions"].tolist() == [[0, 3, 2], [2, 0, 0], [0, 2, 2]]
    assert da["contigs"][:, 0].tolist() == [100, 140, 300, 333] and da["contigs"][:, -1].tolist() == [0, -1, 1, 2]
    assert da["alignments"][:, -1].tolist() == [0, 2, 3]   # the contig of each alignment, in caller order
    assert da["cigar"].ravel().tolist() == [0x50, 0x21, 0x30, 0x40, 0x12, 0x31]
    assert bytes(da["contig_bases"].astype(np.uint8)) == b"ACGTAGGCTTACCAGGTT"
    assert da["events"][:, 0].tolist() == [0, 0, 2] and da["events"][:, -4:-2].tolist() == [[1 << 18, 7], [0, 12], [0, 99]]


def test_dump_samples_a_large_table(monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SHARE", 40)
    r = [results(True)]
    d = bench.dump_results(r)
    rows = d["contig_bases_rows"].astype(np.int64)
    assert 0 < len(rows) < 18 and np.all(np.diff(rows) > 0)
    assert bytes(d["contig_bases"].astype(np.uint8)) == bytes(np.frombuffer(b"ACGTAGGCTTACCAGGTT", np.uint8)[rows])
    for k in ("regions", "contigs", "alignments", "cigar", "events", "contig_bases"):
        assert d[k].nbytes + (d[k + "_rows"].nbytes if k + "_rows" in d else 0) <= 40, k
    assert np.array_equal(bench.dump_results(r)["contig_bases_rows"], d["contig_bases_rows"])   # the same sample every time


@pytest.mark.gpu
def test_two_runs_dump_the_same_outputs(tmp_path):
    dumps = []
    for i in range(2):
        out = tmp_path / str(i)
        subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--scale", "0.02", "--cpu-sample", "100",
                        "--no-bam-leg", "--dump-outputs", str(out)], check=True, capture_output=True, timeout=900)
        dumps.append({f: np.load(out / f) for f in sorted(os.listdir(out))})
    assert sorted(dumps[0]) == sorted(dumps[1]) and "events.npy" in dumps[0] and dumps[0]["counts.npy"][0] > 0
    assert sum(a.nbytes for a in dumps[0].values()) <= bench.DUMP_BYTES
    for k, a in dumps[0].items():
        assert np.array_equal(a, dumps[1][k]), k
