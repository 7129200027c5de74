"""Reverse-mode user densities compile without a GPU: every log_density source of the tests and the README gets
through NVRTC with the reverse-mode header at small and large dims and fails only at loading the code (no device
here).  On a GPU box the same sources run (tests/test_gpu_user_model_reverse.py)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GOOD_AD = """template <typename S, typename T> __device__ S log_density(const S* q, int d, const T* data) {
        S lp = (T)0; for (int i = 0; i < d; ++i) lp -= softplus(q[i]) + square(q[i]) * exp(-q[0]) / (T)3 + log1p(square(q[i])); return lp; }"""

# every operator and function of the header, and a branch on the value (.v), as a source may use them
ALL_OPS = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data) {
    S lp = S(0.0, 0);
    for (int i = 0; i < d; ++i) {
        S a = q[i], b = q[(i + 1) % d];
        S t = a + b - a * b / (b * b + (T)1) + (-a);
        t += a; t -= b; t += (T)1; t -= (T)2;
        t = t + (T)1 - (T)3 * t / (T)4 + (T)2 * t - (T)1 / (square(t) + (T)1) + ((T)1 - t) - t * (T)0.5;
        if (a.v > (T)0) t = t + log(a + (T)1) + pow(a + (T)1, (T)1.5) + sqrt(a + (T)1);
        lp -= exp(-square(t)) + log1p(square(a)) + tanh(t) + sin(a) * cos(b) + softplus(t);
    }
    return lp;
}
"""


def _sources():
    import importlib.util
    spec = importlib.util.spec_from_file_location("um", os.path.join(ROOT, "tests", "test_gpu_user_model.py"))
    text = open(spec.origin).read()
    found = dict(re.findall(r'^(FUNNEL_DENSITY|LOGISTIC_DENSITY) = r"""(.*?)"""', text, flags=re.M | re.S))
    nuts = open(os.path.join(ROOT, "tests", "test_gpu_nuts.py")).read()
    iid = re.search(r'src = r?"""(\s*template <typename S, typename T>.*?)"""', nuts, flags=re.S)
    readme = open(os.path.join(ROOT, "README.md")).read()
    funnel = re.search(r"UserModel\(r'''(.*?)'''", readme, flags=re.S)
    assert set(found) == {"FUNNEL_DENSITY", "LOGISTIC_DENSITY"} and iid and funnel
    return {"funnel": found["FUNNEL_DENSITY"], "logistic": found["LOGISTIC_DENSITY"], "iid": iid.group(1),
            "readme": funnel.group(1), "good_ad": GOOD_AD, "all_ops": ALL_OPS}


@pytest.fixture(scope="module")
def lib():
    import torch
    if torch.cuda.is_available():
        pytest.skip("meant for machines without a GPU")
    from aehmc_b200 import _lib
    lib = _lib.load()
    lib.b2h_last_error.restype = C.c_char_p
    return lib


def _create(lib, src, dim):
    h = C.c_void_p()
    rc = lib.b2h_user_model_create_rev(src.encode(), C.c_int32(dim), C.byref(h))
    msg = lib.b2h_last_error().decode()
    if "libnvrtc" in msg:
        pytest.skip("NVRTC is not installed on this machine")
    return rc, msg


@pytest.mark.parametrize("dim", [1, 65, 1000])
@pytest.mark.parametrize("name", ["funnel", "logistic", "iid", "readme", "good_ad", "all_ops"])
def test_reverse_sources_compile(lib, name, dim):
    rc, msg = _create(lib, _sources()[name], dim)
    assert rc != 0 and "loading" in msg, msg


def test_reverse_compile_error_reports_the_log(lib):
    rc, msg = _create(lib, "template <typename S, typename T> __device__ S log_density(const S* q, int d, const T* data) "
                           "{ return undefined_symbol; }", 70)
    assert rc != 0 and "does not compile" in msg and "undefined_symbol" in msg, msg


@pytest.mark.parametrize("dim", [0, -1, 4097])
def test_reverse_dim_is_checked(lib, dim):
    rc, msg = _create(lib, GOOD_AD, dim)
    assert rc != 0 and "dim must be" in msg, msg
