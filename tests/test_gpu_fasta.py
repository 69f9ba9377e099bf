"""A bgzip-compressed reference inflated and parsed on the device (idl_fasta_open): byte for byte the host loader's names and sequences, the same
errors, the same batches through idl_bam_set_reference_fasta, and the same VCF from every front end as with the plain FASTA."""
import os
import subprocess

import numpy as np
import pytest

from indelope_b200 import abi, api, build, cuda, host
import fasta_corpus as fc
import idl_testutil as util

pytestmark = pytest.mark.gpu
CALL = dict(min_reads=5, min_ctg_len=73, min_event_len=5)


def _host(path):
    names, seqs = host.Dataset.load_fasta(path).sequences()
    return names, [bytes(s) for s in seqs]


def _device(data):
    f = cuda.Fasta(data)
    try:
        out = (f.names, [bytes(f.sequence(r)) for r in range(f.n_records)])
        assert f.lengths == [len(s) for s in out[1]] and f.info["sequence_bytes"] == sum(f.lengths)
        return out
    finally:
        f.close()


def test_corpus_equals_the_host_parse(tmp_path):
    n = 0
    for name, text in fc.corpus().items():
        for block in fc.member_sizes(text):
            data = fc.bgzf(text, block)
            p = tmp_path / "c.fa.gz"
            p.write_bytes(data)
            assert _device(data) == _host(str(p)), (name, block)
            n += 1
    assert n > 100


def test_boundary_lengths_and_tiles(tmp_path):
    """texts of every length mod 4 and with '\\n', '\\r', '>' and name ends on the parse's 8 KiB tiles and 32-byte thread slices"""
    rng = np.random.default_rng(3)
    texts = []
    for L in list(range(1, 70)) + [8190, 8191, 8192, 8193, 8194, 8195, 16383, 16384, 16385, 3 * 8192 + 2]:
        body = bytearray(rng.choice(list(b"ACGTacgtN \r\n"), size=L).astype(np.uint8).tobytes())
        body[0:1] = b">"
        texts.append(bytes(body))
    for edge in (32, 8192, 2 * 8192, 5 * 8192):
        for d in range(-3, 4):
            for put in (b"\n", b"\r\n", b"\n>", b" \n", b"\r", b"\n\n>x y\n", b"\t"):
                t = bytearray(fc.wrap(bytes(rng.choice(list(b"ACGT"), size=6 * 8192).astype(np.uint8).tobytes()), 77))
                t[0:4] = b">a b"
                at = edge + d
                t[at:at + len(put)] = put
                texts.append(bytes(t))
    for k, t in enumerate(texts):
        data = fc.bgzf(t, 4096 if k % 2 else 61)
        p = tmp_path / "b.fa.gz"
        p.write_bytes(data)
        assert _device(data) == _host(str(p)), k


@pytest.mark.parametrize("name", ["unwrapped_50mb", "wrapped_2x40mb"])
def test_large_references(tmp_path, name):
    text = fc.large(name)
    data = fc.bgzf(text, 0xff00, levels=((1, 0),))
    p = tmp_path / "l.fa.gz"
    p.write_bytes(data)
    f = cuda.Fasta(data)
    try:
        want = fc.parse(text)
        assert f.names == [n for n, _ in want]
        for r, (_, s) in enumerate(want):
            assert bytes(f.sequence(r)) == s, r
        assert f.info["inflated_bytes"] == len(text) and f.info["parse_algorithmic_bytes"] >= len(text)
    finally:
        f.close()
    assert _host(str(p)) == ([n for n, _ in want], [s for _, s in want])


@pytest.mark.parametrize("case", sorted(fc.errors()))
def test_errors_match_the_host(tmp_path, case):
    data, phrase = fc.errors()[case]
    p = tmp_path / "e.fa.gz"
    p.write_bytes(data)
    with pytest.raises(IOError, match=phrase.replace("'", ".")):
        host.Dataset.load_fasta(str(p))
    with pytest.raises(cuda.IdlError, match=phrase.replace("'", ".")):
        cuda.Fasta(data)


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """the regions fixture of test_gpu_regions.py (two ~400 kb targets), its FASTA also bgzipped with a member boundary exactly on the second
    record's '>'"""
    d = tmp_path_factory.mktemp("fagz_gpu")
    ds = util.small_dataset("pr1", chrom_len=400_000, n_events=60, max_indel=40, n_chroms=2, n_base_rate=0.0005, dup_fraction=0.02)
    fa, gz, bam = str(d / "ref.fa"), str(d / "ref.fa.gz"), str(d / "reads.bam")
    ds.write_fasta(fa)
    ds.write_bam(bam, level=1)
    text = open(fa, "rb").read()
    cut = text.index(b"\n>") + 1
    open(gz, "wb").write(fc.bgzf_cut(text, [cut]))
    return ds, fa, gz, bam, d


def test_member_boundary_on_a_record(files):
    ds, fa, gz, bam, d = files
    f = cuda.Fasta(open(gz, "rb").read())
    assert f.names == ["chrS1", "chrS2"] and f.info["n_members"] > 2
    f.close()


def test_placement_gives_the_same_batch(files):
    """idl_bam_pack after idl_bam_set_reference_fasta == after idl_bam_set_reference with the host's sequence, all four pools"""
    from test_gpu_bam import _batch_bytes
    ds, fa, gz, bam, d = files
    data = open(bam, "rb").read()
    rois = host.Dataset.load(fa, bam).sweep(min_reads=5)
    a = rois.arrays()
    n = rois.n_rois
    params = abi.default_params(**CALL)
    ctx = cuda.Context(0, params)
    f = cuda.Fasta(open(gz, "rb").read())
    b1, b2 = cuda.Bam(data), cuda.Bam(data)
    nr, sb, rb = rois.pack_size(0, n, params)
    out = []
    for b, place in ((b1, lambda b, c: b.set_reference(c, a["chrom_seqs"][c])), (b2, lambda b, c: b.set_reference_fasta(c, f, f.names.index(b.ref_names[c])))):
        for c in range(b.n_ref):
            place(b, c)
        batch = ctx.batch_alloc(n + 8, nr + 8, sb + 64, rb + 64)
        ctx.bam_pack(b, a["roi_chrom"], a["roi_start"], a["roi_stop"], a["roi_n_reads"], a["read_idx"], batch)
        out.append(_batch_bytes(batch))
        ctx.batch_free(batch)
    for k in ("sizes", "summary", "region", "read", "seq2", "seqn", "ref2", "refn"):
        assert out[0][k] == out[1][k], k
    small = cuda.Fasta(util.bgzf_compress(b">chrS1\nACGT\n"))
    with pytest.raises(cuda.IdlError):
        b1.set_reference_fasta(0, small, 0)   # a length that is not the target's
    b1.close(); b2.close(); f.close(); small.close(); ctx.close()


def _cli(args, fa, bam, env=None):
    exe = build.build_cli()
    opts = ["--min-reads", "5", "--min-contig-len", "73", "--min-event-len", "5"]
    return subprocess.run([exe] + opts + args + [fa, bam], capture_output=True, text=True, env=dict(os.environ, INDELOPE_TIMING="1", **(env or {})))


def test_front_ends_give_the_same_vcf(files):
    ds, fa, gz, bam, d = files
    bed = str(d / "r.bed")
    open(bed, "w").write("chrS1\t100000\t180000\nchrS2\t0\t50000\nchrS2\t390000\t400000\n")
    n_calls = 0
    for args, env in (([], None), (["-g"], None), (["-g"], {"INDELOPE_BY_TARGET": "1"}), (["-r", "chrS1:200,001-260,000", "-r", "chrS2:5000-90000"], None),
                      (["-R", bed], None), (["-g", "-R", bed], None)):
        r1, r2 = _cli(args, fa, bam, env), _cli(args, gz, bam, env)
        assert r1.returncode == 0 and r2.returncode == 0, (args, r1.stderr, r2.stderr)
        assert r1.stdout == r2.stdout, (args, util.diff_lines(r1.stdout, r2.stdout))
        n_calls += r1.stdout.count("\n") - r1.stdout.count("#")
        if "-g" in args or "-R" in args or "-r" in args:
            assert "reference on the device" in r2.stderr, r2.stderr
    assert n_calls > 10
    for kw in ({}, {"by_target": True}, {"regions": ["chrS1:200,001-260,000"], "bed": bed}):
        assert api.call_bam(fa, bam, max_reads=3000, **kw, **CALL) == api.call_bam(gz, bam, max_reads=3000, **kw, **CALL), kw


def test_front_end_errors_leave_stdout_empty(files, tmp_path):
    ds, fa, gz, bam, d = files
    import gzip
    plain = tmp_path / "plain.fa.gz"
    plain.write_bytes(gzip.compress(open(fa, "rb").read()))
    bad = tmp_path / "bad.fa.gz"
    bad.write_bytes(util.bgzf_compress(b"ACGT\n" + open(fa, "rb").read()))
    for path, msg in ((str(plain), "bgzip"), (str(bad), "does not start with")):
        for args, env in (([], None), (["-g"], None), (["-g"], {"INDELOPE_BY_TARGET": "1"}), (["-r", "chrS1:1-100"], None)):
            r = _cli(args, path, bam, env)
            assert r.returncode == 1 and r.stdout == "" and msg in r.stderr, (path, args, r.stderr)
