"""A bgzip-compressed reference (ref.fa.gz) on the host: every loader of libindelope_host inflates its BGZF members and parses the text by the rules of
the plain loader, so a .fa.gz gives the same names, sequences, datasets and regions as the .fa; plain gzip and corrupt members are refused."""
import os
import subprocess

import numpy as np
import pytest

from indelope_b200 import build, host
import fasta_corpus as fc
import idl_testutil as util


def _sequences(path):
    names, seqs = host.Dataset.load_fasta(path).sequences()
    return names, [bytes(s) for s in seqs]


def test_rules_model_matches_the_plain_loader(tmp_path):
    """the Python statement of the rules (fasta_corpus.parse) is what the plain loader does, so it can describe the corpus"""
    for name, text in fc.corpus().items():
        p = tmp_path / (name + ".fa")
        p.write_bytes(text)
        want = fc.parse(text)
        assert _sequences(str(p)) == ([n for n, _ in want], [s for _, s in want]), name


def test_bgzipped_corpus_equals_the_plain_file(tmp_path):
    n_files = 0
    for name, text in fc.corpus().items():
        plain = tmp_path / (name + ".fa")
        plain.write_bytes(text)
        want = _sequences(str(plain))
        for k, block in enumerate(fc.member_sizes(text)):
            gz = tmp_path / ("%s.%d.fa.gz" % (name, block))
            gz.write_bytes(fc.bgzf(text, block, levels=fc.LEVELS[k % len(fc.LEVELS):] + fc.LEVELS[:k % len(fc.LEVELS)]))
            assert _sequences(str(gz)) == want, (name, block)
            n_files += 1
    assert n_files > 100


def test_member_edges_inside_headers_and_line_ends(tmp_path):
    """member boundaries on '>', between '\\r' and '\\n', inside a name and inside a trailing run"""
    text = b">first one\r\nACGT  \r\nAC\r\n>second\tx\r\n\r\nGGG \r \n>third"
    for cut in range(1, len(text)):
        gz = tmp_path / "cut.fa.gz"
        gz.write_bytes(fc.bgzf_cut(text, [cut]))
        want = fc.parse(text)
        assert _sequences(str(gz)) == ([n for n, _ in want], [s for _, s in want]), cut


def test_threads_do_not_change_the_result(tmp_path):
    text = fc.corpus()["many_records"]
    gz = tmp_path / "t.fa.gz"
    gz.write_bytes(fc.bgzf(text, 61))
    try:
        host.set_threads(1)
        one = _sequences(str(gz))
        host.set_threads(7)
        assert _sequences(str(gz)) == one
    finally:
        host.set_threads(0)


@pytest.mark.parametrize("case", sorted(fc.errors()))
def test_errors_are_refused_with_their_message(tmp_path, case):
    data, phrase = fc.errors()[case]
    p = tmp_path / (case + ".fa.gz")
    p.write_bytes(data)
    with pytest.raises(IOError, match=phrase.replace("'", ".")):
        host.Dataset.load_fasta(str(p))


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """the test_files dataset, its FASTA written plain and bgzipped (a member boundary exactly on the second record's '>')"""
    d = tmp_path_factory.mktemp("fagz")
    ds = util.small_dataset("pr1", chrom_len=120_000, n_events=24, max_indel=40, n_chroms=2, n_base_rate=0.0005, dup_fraction=0.02)
    fa, gz, bam = str(d / "ref.fa"), str(d / "ref.fa.gz"), str(d / "reads.bam")
    ds.write_fasta(fa)
    ds.write_bam(bam, level=1)
    text = open(fa, "rb").read()
    open(gz, "wb").write(fc.bgzf_cut(text, [text.index(b"\n>") + 1]))
    return ds, fa, gz, bam


def _view(rois):
    a = rois.arrays()
    return {k: (list(v) if k == "chrom_names" else [bytes(x) for x in v] if k == "chrom_seqs" else np.asarray(v).tobytes()) for k, v in a.items()}


def test_same_datasets_from_fa_and_fa_gz(files):
    ds, fa, gz, bam = files
    assert _view(host.Dataset.load(fa, bam, threads=2).sweep(min_reads=5)) == _view(host.Dataset.load(gz, bam, threads=2).sweep(min_reads=5))
    g1 = [_view(g) for g in host.Stream(fa, bam, min_reads=5).groups(100)]
    g2 = [_view(g) for g in host.Stream(gz, bam, min_reads=5).groups(100)]
    assert g1 == g2 and len(g1) > 1
    for target, beg, end in (("chrS1", 0, 0), ("chrS2", 30_000, 61_000)):
        r1 = host.Dataset.load_region(fa, bam, target, beg, end).sweep(min_reads=5)
        r2 = host.Dataset.load_region(gz, bam, target, beg, end).sweep(min_reads=5)
        assert _view(r1) == _view(r2)
    t = host.Dataset.load_fasta(gz)
    t.set_bam_targets(bam)
    assert t.sequences()[0] == ["chrS1", "chrS2"]


def test_dataset_from_sequences(files):
    ds, fa, gz, bam = files
    names, seqs = host.Dataset.load_fasta(fa).sequences()
    d = host.Dataset.from_sequences(list(reversed(names)), [bytes(s) for s in reversed(seqs)])
    d.set_bam_targets(bam)
    n2, s2 = d.sequences()
    assert n2 == names and [bytes(x) for x in s2] == [bytes(x) for x in seqs]


def test_cli_with_fa_gz_and_no_device(files):
    if util.has_gpu():
        pytest.skip("GPU present")
    ds, fa, gz, bam = files
    exe = build.build_cli()
    for args in ([], ["-g"]):
        r = subprocess.run([exe, "--min-reads", "5"] + args + [gz, bam], capture_output=True, text=True)
        assert r.returncode == 1 and r.stdout == "" and "no CPU path" in r.stderr, (args, r.stderr)
    bad = os.path.join(os.path.dirname(gz), "plain.fa.gz")
    import gzip
    open(bad, "wb").write(gzip.compress(open(fa, "rb").read()))
    r = subprocess.run([exe, bad, bam], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == "" and "bgzip" in r.stderr, r.stderr
