"""Regenerate tests/golden/* from the CPU oracle (the fixtures are committed).

  python tools/make_golden.py               # pr1_small, tandem_small
  python tools/make_golden.py --lane-fuzz   # ksw2_lane_fuzz.npz: only with oracle/_ref built (see make_lane_fuzz)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from indelope_b200 import host  # noqa: E402
from oracle import pyoracle as orc  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


FIXTURES = {
    # BASELINE config 1 in small
    "pr1_small": dict(chrom_len=300_000, n_events=60),
    # tandem-repeat rich: most events fall back to the two unbanded alignments per read (src/indelope.nim:312-372)
    "tandem_small": dict(chrom_len=300_000, n_events=60, max_indel=40, tr_fraction=0.8, tr_max_unit=4, seed=31),
}


def main():
    os.makedirs(GOLD, exist_ok=True)
    if "--lane-fuzz" in sys.argv:
        return make_lane_fuzz()
    for name, over in FIXTURES.items():
        make(name, over)


def make_lane_fuzz():
    """the lane model's fields and full CIGAR on the pairs of test_lane_model_equals_compiled_reference_fuzz.  These vectors keep the lane
    model where it was when it matched the compiled reference; rewriting them without that reference would move them to whatever the
    lane model computes now, so this refuses unless oracle/_ref is built, and checks every pair against it before writing."""
    from test_oracle_ksw2 import lane_fuzz_pairs, pairs_digest
    if not orc.have_ref():
        sys.exit("tests/golden/ksw2_lane_fuzz.npz is only rewritten after checking the lane model against the compiled reference: build oracle/_ref first")
    pairs = lane_fuzz_pairs()
    fields, cigars = [], []
    for it, (q, t, go, w, z) in enumerate(pairs):
        f, c, _ = orc.ksw2(q, t, gapo=go, gape=1, w=w, zdrop=z, impl="lane")
        assert orc.ksw2(q, t, gapo=go, gape=1, w=w, zdrop=z, impl="ref")[:2] == (f, c), ("lane model and compiled reference DP disagree", it)
        fields.append([f[k] for k in orc.EZ_FIELDS]); cigars.append(c)
    cigar = np.array([x for c in cigars for x in c], dtype=np.uint32)  # pair i's ops follow those of pairs < i (n_cigar of each)
    np.savez_compressed(os.path.join(GOLD, "ksw2_lane_fuzz.npz"), inputs_sha256=np.array(pairs_digest(pairs)), fields=np.array(fields, dtype=np.int32),
                        cigar=cigar, made_with=np.array("lane"))
    print("ksw2_lane_fuzz: %d pairs, %d CIGAR ops, equal to the compiled reference" % (len(pairs), len(cigar)))


def make(name, over):
    cfg = dict(host.CONFIGS["pr1"]); cfg.update(over)
    ds = host.Dataset(**cfg)
    rois = ds.sweep(min_reads=5)
    use_ref = orc.have_ref()
    dump, vcf, cnt = orc.call(rois.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, use_ref_ksw2=use_ref, dump_level=31)
    d2, v2, _ = orc.call(rois.arrays(), min_reads=5, min_ctg_len=73, min_event_len=5, use_ref_ksw2=False, dump_level=31)
    assert (dump, vcf) == (d2, v2), "lane model and compiled reference DP disagree"
    with open(os.path.join(GOLD, name + ".vcf"), "w") as f:
        f.write(rois.header() + vcf)
    with open(os.path.join(GOLD, name + ".dump"), "w") as f:
        f.write("\n".join(l for l in dump.splitlines() if l[:1] in "RAEV") + "\n")
    print(name, "regions", cnt["regions"], "AL events", cnt["al_events"], "unbanded alignments", cnt["dp_b"], "variants", cnt["variants"], "reference ksw2 used:", use_ref)


if __name__ == "__main__":
    main()
