"""CPU-side checks of the drop-in boundary: the shared library loads without a GPU, exports every symbol
that include/b200hmc.h declares, and refuses to run without a CUDA device (no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "aehmc_b200", "lib", "libb200hmc.so")
HEADER = os.path.join(ROOT, "include", "b200hmc.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b2h_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import __graft_entry__
        __graft_entry__.build()
    return ctypes.CDLL(LIB)


def test_header_symbols_are_exported(lib):
    names = _declared()
    assert len(names) >= 24
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_python_binding_lists_the_same_symbols():
    from aehmc_b200 import _lib
    assert sorted(_lib.EXPORTS) == _declared()


def test_struct_layouts_match_header_sizes(tmp_path):
    """ctypes mirrors of the C structs have the sizes gcc gives include/b200hmc.h."""
    import shutil
    import subprocess
    from aehmc_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("needs gcc")
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "b200hmc.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n", '
                   'sizeof(b2h_model), sizeof(b2h_metric), sizeof(b2h_rng), sizeof(b2h_diag), sizeof(b2h_adapt), '
                   'sizeof(b2h_cfg), sizeof(b2h_gemm_group)); return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    mine = [ctypes.sizeof(getattr(_lib, n)) for n in ("Model", "Metric", "Rng", "Diag", "Adapt", "Cfg", "GemmGroup")]
    assert mine == sizes


def test_version_and_error_string(lib):
    lib.b2h_last_error.restype = ctypes.c_char_p
    assert lib.b2h_version() == 100
    assert isinstance(lib.b2h_last_error(), bytes)


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib.b2h_last_error.restype = ctypes.c_char_p
    handle = ctypes.c_void_p()
    rc = lib.b2h_ctx_create(0, None, ctypes.byref(handle))
    assert rc != 0 and b"no CPU fallback" in lib.b2h_last_error()
    import aehmc_b200
    from aehmc_b200._lib import B200HMCError
    with pytest.raises(B200HMCError):
        aehmc_b200.models.NealFunnel(10)


def test_product_does_not_import_the_oracle():
    """The oracle is test infrastructure: nothing under aehmc_b200/ may reference it."""
    pkg = os.path.join(ROOT, "aehmc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "host_sim" not in text, f


def test_user_model_sources_compile_without_a_gpu():
    """NVRTC needs no device: a valid user source (hand-written gradient, or density-only with the forward-mode dual
    header) gets through compilation and fails only at loading the code (no GPU here); a broken one reports the
    compiler log.  On a GPU box the same calls succeed (tests/test_gpu_user_model.py)."""
    import ctypes as C
    import torch
    if torch.cuda.is_available():
        pytest.skip("meant for machines without a GPU")
    from aehmc_b200 import _lib
    lib = _lib.load()
    good = b"""template <typename T> __device__ T potential_and_grad(const T* q, T* g, int d, const T* data) {
        T U = 0; for (int i = 0; i < d; ++i) { U += (T)0.5 * q[i] * q[i]; g[i] = q[i]; } return U; }"""
    good_ad = b"""template <typename S, typename T> __device__ S log_density(const S* q, int d, const T* data) {
        S lp = (T)0; for (int i = 0; i < d; ++i) lp -= softplus(q[i]) + square(q[i]) * exp(-q[0]) / (T)3 + log1p(square(q[i])); return lp; }"""
    h = C.c_void_p()
    for call, text in ((lambda: lib.b2h_user_model_create(good, C.byref(h)), "loading"),
                       (lambda: lib.b2h_user_model_create_ad(good_ad, C.c_int32(6), C.byref(h)), "loading"),
                       (lambda: lib.b2h_user_model_create(b"this is not CUDA", C.byref(h)), "does not compile"),
                       (lambda: lib.b2h_user_model_create_ad(good_ad, C.c_int32(1000), C.byref(h)), "dim must be")):
        assert call() != 0
        msg = lib.b2h_last_error().decode()
        if "libnvrtc" in msg:
            pytest.skip("NVRTC is not installed on this machine")
        assert text in msg, msg
