"""CPU tests of the product's host side: the C-ABI library loads without a GPU, exports every symbol
include/rnnoise.h declares, parses models exactly like the reference, and refuses to run without CUDA."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np

import nnnoiseless_b200 as nb
import oracle
from conftest import ROOT


def test_header_symbols_exported():
    hdr = open(os.path.join(ROOT, "include", "rnnoise.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(rnnoise_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(nb.C_ABI_SYMBOLS)
    L = nb.lib()
    for sym in declared:
        assert getattr(L, sym) is not None


def test_reference_abi_basics():
    L = nb.lib()
    assert L.rnnoise_get_frame_size() == 480  # src/capi.rs:17-19
    assert L.rnnoise_get_size() > 0


def _mutations(good: bytes):
    yield good[:-1]                      # truncated
    yield good + b"\x00"                 # trailing byte (src/rnn.rs:196-198)
    yield b""                            # empty
    yield b"\x2a\x18"                    # short header
    bad = bytearray(good); bad[0] = 41; yield bytes(bad)          # input_dense.ni != 42
    bad = bytearray(good); bad[2] = 3; yield bytes(bad)           # unknown activation
    bad = bytearray(good); bad[1] = 0x80; yield bytes(bad)        # negative neuron count
    bad = bytearray(good); bad[1035 + 1] = 25; yield bytes(bad)   # vad_gru.nn changes -> sizes no longer chain


def test_model_parser_matches_oracle(builtin_bytes, sh_bytes):
    for good in (builtin_bytes, sh_bytes):
        m = nb.RnnModel.from_bytes(good)
        assert m is not None and m.to_bytes() == good and oracle.model_accepts(good)
        for bad in _mutations(good):
            assert nb.RnnModel.from_bytes(bad) is None
            assert not oracle.model_accepts(bad)


def test_builtin_model_is_weights_rnn(builtin_bytes):
    assert nb.RnnModel().to_bytes() == builtin_bytes and len(builtin_bytes) == 87521


def test_text_model_conversion(sh_bytes):
    """N3 (train/convert_rnnoise.py:18-29): the reference's own text fixture test_data/sh.rnnn (committed as
    tests/golden/sh.rnnn) through rnnoise_model_from_text equals the image the independent restatement of the
    converter (tests/golden/make_sh_rnn.py) produces from it, byte for byte."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_sh_rnn", os.path.join(ROOT, "tests", "golden", "make_sh_rnn.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    text = open(os.path.join(ROOT, "tests", "golden", "sh.rnnn")).read()
    assert gen.convert(text) == sh_bytes and len(sh_bytes) == 87521  # the committed binary fixture is the generator's output
    m = nb.RnnModel.from_text(text)
    assert m is not None and m.to_bytes() == sh_bytes
    assert oracle.model_accepts(sh_bytes)
    # negative numbers wrap like python's int(s) % 256; junk is rejected
    assert nb.RnnModel.from_text("wrong header\n1 2 3") is None
    assert nb.RnnModel.from_text("rnnoise-nu model file version 1\n1 2 x") is None
    assert nb.RnnModel.from_text(text[: len(text) // 2]) is None  # truncated image no longer chains (src/rnn.rs:196-222)


def test_model_from_file_takes_over_file(tmp_path, builtin_bytes):
    p = tmp_path / "m.rnn"
    p.write_bytes(builtin_bytes)
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    f = libc.fopen(str(p).encode(), b"rb")
    h = nb.lib().rnnoise_model_from_file(f)  # closes f (src/capi.rs:93-94)
    assert h
    nb.lib().rnnoise_model_free(h)
    p.write_bytes(builtin_bytes[:100])
    f = libc.fopen(str(p).encode(), b"rb")
    assert not nb.lib().rnnoise_model_from_file(f)


def test_no_cpu_fallback():
    """Without a visible CUDA device the constructors raise; a child process with every GPU hidden checks this on a
    machine that has one too."""
    code = ("import pytest\n"
            "import nnnoiseless_b200 as nb\n"
            "with pytest.raises(nb.NnnoiselessError, match='no CUDA device'):\n"
            "    nb.DenoiseBatch(4)\n"
            "with pytest.raises(nb.NnnoiselessError):\n"
            "    nb.DenoiseState()\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "nnnoiseless_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(dirpath, fn), errors="replace").read()
                assert "import oracle" not in txt and "nno_oracle" not in txt and "from oracle" not in txt, fn


def test_shard_streams_partition():
    for n, w in [(262144, 8), (65536, 3), (5, 8), (37, 4)]:
        spans = [nb.shard_streams(n, w, r) for r in range(w)]
        assert spans[0][0] == 0 and sum(c for _, c in spans) == n
        for (s0, c0), (s1, _) in zip(spans, spans[1:]):
            assert s0 + c0 == s1


def test_model_parser_fuzz_agrees_with_oracle(builtin_bytes):
    """Loader hardening (SURVEY 8(f) N3): on mutated / truncated / extended model images the product's parser and the
    oracle's restatement of RnnModel::from_bytes (src/rnn.rs:116-232) accept exactly the same inputs, and an
    accepted image round-trips byte for byte."""
    from hypothesis import given, settings, strategies as st

    good = builtin_bytes
    # header bytes of the six layers (ni, nn, activation): the interesting places to corrupt
    offs = [0, 1035, 4566, 24585, 85356, 87493]
    hdr = [o + k for o in offs for k in range(3)]

    @settings(max_examples=150, deadline=None)
    @given(st.lists(st.tuples(st.sampled_from(hdr) | st.integers(0, len(good) - 1), st.integers(0, 255)), min_size=0, max_size=3),
           st.integers(-40, 40))
    def check(edits, dlen):
        b = bytearray(good)
        for pos, val in edits:
            b[pos] = val
        b = bytes(b[:len(b) + dlen]) if dlen < 0 else bytes(b) + bytes(dlen)
        ours = nb.RnnModel.from_bytes(b)
        assert (ours is not None) == oracle.model_accepts(b)
        if ours is not None:
            assert ours.to_bytes() == b

    check()


def test_tcgen05_weight_packing_selftest(builtin_bytes, sh_bytes):
    """The tcgen05 GRU kernel's model image (K-major UMMA operands per layer phase, activation-chunk lists, biases) replayed
    on the host in plain f32 equals a direct evaluation of src/rnn.rs:343-379 from the model bytes -- the packing logic is
    checked without a GPU (the instruction / TMEM layouts themselves: tools/probes/tcgen05_probe.cu on the GPU)."""
    L = nb.lib()
    L.nnb_tc_pack_selftest.restype = C.c_double
    L.nnb_tc_pack_selftest.argtypes = [C.c_char_p, C.c_size_t, C.c_int]
    for model in (builtin_bytes, sh_bytes):
        for seed in range(8):
            assert 0.0 <= L.nnb_tc_pack_selftest(model, len(model), seed) < 2e-5
    assert L.nnb_tc_pack_selftest(builtin_bytes[:-1], len(builtin_bytes) - 1, 0) == -1.0


def test_bench_reads_measured_traffic_of_every_kernel():
    """bench.py's roofline.traffic comes from the newest committed `ncu --set full` raw page under profiles/: the page
    must hold the five kernels of a frame-step under the names bench.py looks for (a renamed kernel would silently turn
    traffic into null), and the dominant kernel's DRAM bytes must stay close to its algorithmic bytes."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    traffic, fname = bench.measured_traffic()
    assert fname is not None, "no profiles/rNN_vMM_ncu_raw_B*.csv committed"
    assert traffic is not None and set(traffic) == set(bench.KERNEL_PATTERNS), (fname, traffic)
    for k, v in traffic.items():
        assert 0 < v < 4 * bench.KERNEL_BYTES[k], (k, v, bench.KERNEL_BYTES[k])
    assert traffic["pitch"] < 1.1 * bench.KERNEL_BYTES["pitch"]  # nothing re-read by the dominant kernel
