"""The directed edge fixtures (idl_testutil.edge_fixtures) on the CPU.  The GPU parity tests of test_gpu_edges.py compare the device with
the oracle on these fixtures; the checks here make sure the oracle, run over them, really takes the paths that exist only at a chromosome
end, a window edge or a contig end, so that the fixtures cannot drift back to easy cases unnoticed.  The BAM written from the same reads
reads back as the same records and regions."""
import numpy as np
import pytest

import idl_testutil as util
from indelope_b200 import host
from oracle import pyoracle as orc

K = 27
EDGE_PARAMS = dict(min_reads=3, min_ctg_len=73, min_event_len=5)


def parse_dump(dump):
    """contig lengths, alignment and event records of a dump_level=31 dump"""
    clen, A, E = {}, [], []
    for l in dump.splitlines():
        f = l.split("\t")
        if f[0] == "C":
            clen[(int(f[1]), int(f[2]))] = int(f[5])
        elif f[0] == "A":
            A.append(dict(region=int(f[1]), ci=int(f[2]), start=int(f[3]), ref_len=int(f[4])))
        elif f[0] == "E":
            E.append(dict(region=int(f[1]), ci=int(f[2]), type=f[4], t_start=int(f[5]), t_stop=int(f[6]), len=int(f[7]), q_start=int(f[8]),
                          q_stop=int(f[9]), reject=int(f[10]), tstart=int(f[11]), qstart=int(f[12]), ref_kmer=f[13], alt_kmer=f[14], aligned=int(f[18])))
    return clen, A, E


@pytest.fixture(scope="module")
def edges():
    fx = util.edge_fixtures()
    _, arrays = util.edge_rois(fx)
    dump, vcf, cnt = orc.call(arrays, dump_level=31, **EDGE_PARAMS)
    return fx, arrays, dump, vcf, cnt


def test_the_oracle_reaches_every_edge_path(edges):
    fx, arrays, dump, vcf, cnt = edges
    clen, A, E = parse_dump(dump)
    chrom_len = [len(s) for s in fx["seqs"]]
    chrom_of = [int(c) for c in arrays["roi_chrom"]]
    assert cnt["vote_invariant_violations"] == 0
    # every reject of the k-mer selection: equal k-mers at q_start 0 / homopolymer (1), low complexity (2), equal twice (3), short (10), window < K (11)
    assert {1, 2, 3, 10, 11} <= {e["reject"] for e in E}, sorted({e["reject"] for e in E})
    # a reference window shorter than K: the contig starts fewer than K bases before the chromosome's end
    assert any(a["ref_len"] < K for a in A)
    assert any(e["reject"] == 11 and e["tstart"] < 0 for e in E)
    # events within K bases of a chromosome's start and of its end
    assert any(e["t_start"] < K for e in E if e["reject"] != 11)
    assert any(chrom_len[chrom_of[e["region"]]] - e["t_start"] <= K and e["reject"] == 0 for e in E)
    # the AL fallback on a contig that runs past its reference window (the read windows are suffixes of a shorter window)
    win = {(a["region"], a["ci"]): a["ref_len"] for a in A}
    assert any(e["aligned"] == 1 and win[(e["region"], e["ci"])] < clen[(e["region"], e["ci"])] for e in E)
    # events at a contig's start, and the second k-mer choice near a contig's end (qend = q_stop + 4 < contig length)
    assert any(e["q_start"] == 0 for e in E)
    assert any(e["reject"] == 0 and e["qstart"] == e["q_stop"] + 4 - K and e["q_stop"] + 4 < clen[(e["region"], e["ci"])] for e in E)
    # the VCF holds records within 100 bp of a chromosome's start and of its end
    recs = [(fx["names"].index(l.split("\t")[0]), int(l.split("\t")[1])) for l in vcf.splitlines()]
    assert any(p <= 100 for _, p in recs) and any(chrom_len[c] - p <= 100 for c, p in recs), recs


def test_a_contig_shorter_than_k_is_rejected_on_the_contig_side(edges):
    """-c below K: a contig shorter than a k-mer is aligned; its alt k-mer would start before the contig (the reference raises there), so the
    event is rejected as IDL_EV_WINDOW with no k-mers, like a reference window shorter than K"""
    fx, arrays, _, _, _ = edges
    dump, _, cnt = orc.call(arrays, min_reads=1, min_ctg_len=20, min_event_len=1, dump_level=31)
    clen, A, E = parse_dump(dump)
    short = [e for e in E if clen[(e["region"], e["ci"])] < K]
    assert short and all(e["reject"] == 11 and e["qstart"] < 0 and e["ref_kmer"] == "." and e["alt_kmer"] == "." for e in short)
    assert cnt["vote_invariant_violations"] == 0


def test_edge_files_read_back_as_the_fixtures(tmp_path):
    """the FASTA + BAM written from the fixtures (soft clips before position 0 and past the end) through the host reader: the same records, and
    the sweep finds regions touching position 0 and the last base of the chromosomes"""
    fx = util.edge_fixtures()
    fa, bam = util.edge_files(fx, tmp_path)
    ds = host.Dataset.load(fa, bam)
    rois = ds.sweep(min_reads=3)
    a = rois.arrays()
    past = 0
    for c, reads in enumerate(fx["reads"]):
        cr = ds.chrom_reads(c)
        assert cr["chrom_len"] == len(fx["seqs"][c])
        assert np.array_equal(cr["start"], [r["start"] for r in reads]) and np.array_equal(cr["stop"], [r["stop"] for r in reads])
        n = a["len"][cr["first_read"]:cr["first_read"] + len(reads)]
        past += int(np.sum(cr["start"] + n > cr["chrom_len"]))      # trailing bases past the chromosome's end (S operations)
    assert past > 0
    lens = np.array([len(s) for s in fx["seqs"]])
    assert np.any(a["roi_start"] == 0)
    assert np.any(a["roi_stop"] >= lens[a["roi_chrom"]] - 1)
