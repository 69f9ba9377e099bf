"""The DEFLATE decoder of inflate_core.cuh (one-lane CPU build) on streams zlib's encoder never writes (tests/deflate_cases.py, written by
tests/deflate_writer.py): zlib, the reference decoder, accepts a stream with the plan's payload and the member's ISIZE if and only if the
decoder returns INF_OK with the same bytes; otherwise the decoder returns the named error.  Every case runs at a word-aligned and at
unaligned offsets on both builds (no ring / 2 KiB ring), and once more under AddressSanitizer laid out as the last member of a file, with
the device's window lookahead loads (IDL_INF_LOOKAHEAD) -- no load may leave the member."""
import ctypes as C
import functools
import hashlib
import json
import os
import pickle
import random
import subprocess
import sys
import zlib

import pytest

import deflate_cases as dc
import deflate_writer as dw

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "indelope_b200", "csrc")
SRC = os.path.join(HERE, "native", "inflate_host.cpp")
OFFSETS = (1, 2, 3, 18, 125)


def _build(out, flags):
    subprocess.check_call(["g++", "-std=c++17", "-fPIC", "-shared", "-Wall", "-x", "c++"] + flags + ["-I", CSRC, SRC, "-o", out])
    lib = C.CDLL(out)
    lib.idl_test_inflate.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_uint32]
    lib.idl_test_inflate_at.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.c_char_p, C.c_uint32]
    lib.idl_test_inflate_tail.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_char_p, C.c_uint32]
    return lib


@pytest.fixture(scope="module", params=[0, 2048], ids=["no-ring", "ring2048"])
def L(request, tmp_path_factory):
    ring = request.param
    return _build(str(tmp_path_factory.mktemp("inflate") / ("libinflate_r%d.so" % ring)), ["-O2", "-DIDL_INF_RING=%d" % ring])


def zlib_ref(stream):
    """zlib's verdict: the output of a complete stream, or None"""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(stream) + d.flush()
    except zlib.error:
        return None
    return out if d.eof and not d.unused_data else None


@functools.lru_cache(maxsize=None)
def corpus():
    """name -> (stream, payload or None, isize, expected decoder results, feature record)"""
    cases = {}
    for k, (name, build) in enumerate(list(dc.VALID.items()) + list(dc.DISTS.items())):
        s, p, F = dw.deflate(build(random.Random(100 + k)))
        cases[name] = (s, p, len(p), {dc.OK}, F)
    for isize in (65535, 65536):
        s, p, F = dw.deflate(dc.stored_65535(random.Random(isize), isize))
        cases["stored_65535_isize_%d" % isize] = (s, p, isize, {dc.OK}, F)
    for name, (plan, expect, isize) in dc.INVALID.items():
        s, p, F = dw.deflate(plan)
        cases[name] = (s, p, F["out_len"] if isize is None else isize, expect, F)
    return cases


def run(L, stream, off, isize):
    out = C.create_string_buffer(isize + 1)
    rc = L.idl_test_inflate(stream, len(stream), out, isize) if off == 0 else L.idl_test_inflate_at(stream, off, len(stream), out, isize)
    return rc, out.raw[:isize]


@pytest.mark.parametrize("name", list(corpus()))
def test_decoder_agrees_with_zlib(L, name):
    stream, payload, isize, expect, _ = corpus()[name]
    ref = zlib_ref(stream)
    accepted = ref is not None and len(ref) == isize
    assert accepted == (dc.OK in expect), "the case is not what it claims to be: zlib %s it" % ("accepts" if accepted else "refuses")
    if accepted:
        assert ref == payload
    for off in (0,) + OFFSETS:
        rc, out = run(L, stream, off, isize)
        if accepted:
            assert rc == dc.OK and out == ref, (off, rc)
        else:
            assert rc in expect, (off, rc, expect)


def _union(names, key):
    out = set()
    for n in names:
        v = corpus()[n][4][key]
        out |= set(v) if isinstance(v, (set, list)) else {v}
    return out


def test_the_corpus_holds_the_constructs():
    """each construct is checked in the streams as written, not in the plans"""
    C_ = corpus()
    valid = [n for n in C_ if dc.OK in C_[n][3]]
    assert _union(valid, "lit_lens_used") == set(range(1, 16))
    assert dw.EOB in _union(valid, "lit_long") and any(s < 256 for s in _union(valid, "lit_long"))
    assert {s for s, l in _union(valid, "len_sym_max_extra") if l >= 11} == set(range(257, 286))
    assert {s for s, l in _union(valid, "dist_long_max_extra") if l >= 9} == set(range(30))
    assert set(range(9, 16)) <= _union(valid, "dist_lens_used")
    for f in ("single_dist_code", "empty_dist_code", "eob_only_code", "rep16_after_zero", "rep18_138", "dist_eq_op"):
        assert True in _union(valid, f), f
    assert {257, 286} <= _union(valid, "hlit") and {1, 30} <= _union(valid, "hdist") and 19 in _union(valid, "hclen")
    assert 7 in _union(valid, "cl_lens_used")
    assert _union(valid, "cross") == {16, 17, 18}
    assert _union(["stored_blocks"], "stored_phases") == set(range(8))
    at = C_["stored_blocks"][4]["stored_data_at"]
    assert {a % 128 for a in at} == set(range(128)) and 0 in C_["stored_blocks"][4]["stored_lens"]
    assert C_["stored_blocks"][4]["blocks"][0] == "stored" and C_["stored_blocks"][4]["stored_lens"][0] == 0    # LEN 0, not final
    assert 65535 in _union(["stored_65535_isize_65535", "stored_65535_isize_65536"], "stored_lens")
    for d in range(1, 41):
        F = C_["dist_%d" % d][4]
        assert F["dists"] == {d} and F["lens"] == set(range(3, 259))
    assert {2047, 2048, 2049, 32768} <= _union(valid, "dists")
    assert {(285, 0), (284, 31)} <= _union(valid, "len_syms")
    F = C_["many_empty_blocks"][4]
    assert F["n_empty_blocks"] >= 1001 and F["blocks"][:1001] == ["fixed"] * 1001 and {"stored", "fixed", "dynamic"} <= set(F["blocks"][1001:])
    # the incomplete codes that must be refused are incomplete, and not the allowed kinds
    assert dw.kraft(dc.INVALID["incomplete_lit"][0][0]["lit"]) < 1 << 15


ASAN_RUNNER = r"""
import ctypes as C, hashlib, json, pickle, sys
lib = C.CDLL(sys.argv[1])
lib.idl_test_inflate_tail.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_char_p, C.c_uint32]
res = []
for name, stream, isize in pickle.load(open(sys.argv[2], "rb")):
    for off in (0, 1, 2, 3, 18):
        for pad in ((-(off + len(stream))) % 4, 8 + 512):
            out = C.create_string_buffer(isize + 1)
            rc = lib.idl_test_inflate_tail(stream, off, len(stream), pad, out, isize)
            res.append([name, off, pad, rc, hashlib.sha1(out.raw[:isize]).hexdigest()])
json.dump(res, sys.stdout)
"""


def test_no_load_leaves_the_member_under_asan(tmp_path):
    """every case laid out as the last member of a file (the stream, then either nothing but the rest of its last word or the 8-byte trailer +
    the 512 zero bytes idl_bam_open puts behind the file), in heap blocks of exactly that size, with the device's window loads"""
    asan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("the compiler has no AddressSanitizer runtime (libasan.so)")
    cases = corpus()
    todo = [(n, c[0], c[2]) for n, c in cases.items()]
    pk = tmp_path / "cases.pkl"
    pk.write_bytes(pickle.dumps(todo))
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1:exitcode=99")
    for ring in (0, 2048):
        so = str(tmp_path / ("libinflate_asan_r%d.so" % ring))
        try:
            subprocess.check_call(["g++", "-std=c++17", "-fPIC", "-shared", "-O1", "-g", "-fsanitize=address", "-fno-omit-frame-pointer", "-x", "c++",
                                   "-DIDL_INF_RING=%d" % ring, "-DIDL_INF_LOOKAHEAD=1", "-I", CSRC, SRC, "-o", so])
        except subprocess.CalledProcessError:
            pytest.skip("the compiler cannot build with -fsanitize=address")
        p = subprocess.run([sys.executable, "-c", ASAN_RUNNER, so, str(pk)], capture_output=True, text=True, env=env, timeout=1200)
        assert p.returncode == 0, "ring %d:\n%s" % (ring, p.stderr[-6000:])
        for name, off, pad, rc, digest in json.loads(p.stdout):
            stream, payload, isize, expect, _ = cases[name]
            assert rc in expect, (name, ring, off, pad, rc)
            if rc == dc.OK:
                assert digest == hashlib.sha1(payload).hexdigest(), (name, ring, off, pad)
