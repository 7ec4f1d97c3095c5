"""The C ABI as seen by real C / C++ clients."""
import os
import subprocess

import numpy as np
import pytest

import nnnoiseless_b200 as nb
from conftest import ROOT, golden_metric

INC = os.path.join(ROOT, "include")
LIBDIR = os.path.dirname(nb.LIB_PATH)


def _cc(args, **kw):
    return subprocess.run(args, capture_output=True, text=True, **kw)


def test_c_client_compiles_and_links(tmp_path):
    exe = tmp_path / "demo_client"
    r = _cc(["gcc", "-std=c99", "-Wall", "-Werror", "-I", INC, os.path.join(ROOT, "tests", "c_client", "demo_client.c"),
             "-o", str(exe), "-L", LIBDIR, "-lnnnoiseless_b200", "-lm", "-Wl,-rpath," + LIBDIR])
    assert r.returncode == 0, r.stderr


def test_cpp_mirror_header_compiles(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "nnnoiseless.hpp"\n'
                   "int main() { auto m = nnnoiseless::RnnModel::from_bytes(nullptr, 0); return m ? 1 : 0; }\n")
    exe = tmp_path / "t"
    r = _cc(["g++", "-std=c++17", "-Wall", "-I", INC, str(src), "-o", str(exe), "-L", LIBDIR, "-lnnnoiseless_b200",
             "-Wl,-rpath," + LIBDIR])
    assert r.returncode == 0, r.stderr
    assert _cc([str(exe)]).returncode == 0  # malformed bytes -> nullopt, no GPU needed


@pytest.mark.gpu
def test_c_client_golden_bytes(tmp_path, reference_output):
    """CI check of the reference (.github/workflows/rust.yml:27-33) restated: the C client's rounded output on
    testing.raw.  Compared with reference_output.raw through the src/lib.rs:184-194 metric (that file was
    written with truncation, the C client rounds: <= 1 LSB apart)."""
    exe = tmp_path / "demo_client"
    r = _cc(["gcc", "-std=c99", "-I", INC, os.path.join(ROOT, "tests", "c_client", "demo_client.c"), "-o", str(exe),
             "-L", LIBDIR, "-lnnnoiseless_b200", "-lm", "-Wl,-rpath," + LIBDIR])
    assert r.returncode == 0, r.stderr
    out = tmp_path / "out.raw"
    r = _cc([str(exe), os.path.join(ROOT, "tests", "golden", "testing.raw"), str(out)])
    assert r.returncode == 0, r.stderr + r.stdout
    got = np.fromfile(out, dtype="<i2")
    assert len(got) == len(reference_output)
    metric, maxdiff = golden_metric([got.astype(np.float32)], reference_output)
    assert metric < 1e-5 and maxdiff <= 1
    # and byte-identical to the batched pcm16 entry point driven with the same frames (B = 1)
    x = np.fromfile(os.path.join(ROOT, "tests", "golden", "testing.raw"), dtype="<i2")[:48000].reshape(100, 1, 480)
    o16, _ = nb.DenoiseBatch(1).process_pcm16_host(x)
    assert np.array_equal(o16[1:].reshape(-1), got)
