"""CPU-only: the C-ABI library loads and exports every symbol include/fastnn.h declares; without a
GPU every compute entry point fails loudly (no CPU fallback)."""
import os
import re

import numpy as np
import pytest

import fastneighbornet_b200 as fnn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    with open(os.path.join(ROOT, "include", "fastnn.h")) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fnn_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    lib = fnn.lib()
    decl = _declared()
    assert len(decl) >= 15
    for s in decl:
        assert hasattr(lib, s), f"{s} declared in include/fastnn.h but not exported"
    assert sorted(fnn.api.ABI_SYMBOLS) == decl


def test_opts_struct_layout():
    o = fnn.default_opts()
    assert (o.mode, o.mult, o.additive, o.canonical_fallback, o.seed, o.use_graph) == (0, 5, 0, 1024, 12345, 1)


def test_trivial_sizes_need_no_device():
    # n <= 3: identity ordering (NetMakerOriginal.java:133-140) - pure host logic
    for n in (1, 2, 3):
        assert fnn.order(np.zeros((n, n))).tolist() == list(range(n + 1))


def test_argument_errors():
    with pytest.raises(fnn.FastNNError) as e:
        fnn.order(None, None, n=5)
    assert e.value.code == -1


@pytest.mark.skipif(fnn.device_count() > 0, reason="GPU present")
def test_fails_loudly_without_gpu():
    with pytest.raises(fnn.FastNNError) as e:
        fnn.order(np.zeros((6, 6)))
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)
    with pytest.raises(fnn.FastNNError):
        fnn.Context(10)


def test_jni_shim_compiles_and_links_against_the_abi(tmp_path):
    """integration/fastnn_jni.c (the reference-side binding of INTEGRATION.md) against a stub jni.h: every libfastnn entry
    point it calls exists with a compatible prototype, and the four natives of integration/NativeNN.java are exported."""
    import subprocess
    so = tmp_path / "libfastnn_jni.so"
    libdir = os.path.dirname(fnn.lib_path())
    cmd = ["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC", "-I", os.path.join(ROOT, "tests", "stubs"), "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "integration", "fastnn_jni.c"), "-L", libdir, "-lfastnn", "-Wl,--no-undefined", "-Wl,--allow-shlib-undefined", "-o", str(so)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    syms = subprocess.run(["nm", "-D", "--defined-only", str(so)], capture_output=True, text=True).stdout
    with open(os.path.join(ROOT, "integration", "NativeNN.java")) as f:
        natives = re.findall(r"static native [\w\[\]]+ (\w+)\(", f.read())
    assert sorted(natives) == ["network", "order", "orderFromFile", "splitWeights"]
    for name in natives:
        assert f"Java_nnet_NativeNN_{name}" in syms


def test_java_patch_applies_to_the_reference(tmp_path):
    """integration/fastnn_java.patch (SURVEY 8f N3: the FastNN.java:326-361, 378/391, 401-466 call-site change plus the seeded
    java.util.Random of NeighborNetLocal.java:30 / NeighborNetRandom.java:27) applies without fuzz to the lines of the
    reference it edits (tests/golden/reference_excerpts: the released v0.3.5 sources around every hunk)."""
    import shutil
    import subprocess
    for f in ("FastNN.java", "NeighborNetLocal.java", "NeighborNetRandom.java"):
        shutil.copy(os.path.join(ROOT, "tests", "golden", "reference_excerpts", f), tmp_path / f)
    r = subprocess.run(["patch", "-p1", "--fuzz=0", "-i", os.path.join(ROOT, "integration", "fastnn_java.patch")], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    src = (tmp_path / "FastNN.java").read_text()
    assert src.count("NativeNN.order(") == 2 and "NativeNN.splitWeights(" in src
