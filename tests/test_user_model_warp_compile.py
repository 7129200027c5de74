"""Warp-form user densities compile without a GPU: every warp-form source of the tests gets through NVRTC for sm_100a
(hand-written and reverse mode, small and large dims) and fails only at loading the code (no device here), and a
thread-form source given to the warp entry point does not compile.  On a GPU box the same sources run
(tests/test_gpu_user_model_warp.py)."""
import ctypes as C

import pytest

import warp_sources
from test_gpu_user_model import BANANA_SRC, FUNNEL_DENSITY


@pytest.fixture(scope="module")
def lib():
    import torch
    if torch.cuda.is_available():
        pytest.skip("meant for machines without a GPU")
    from aehmc_b200 import _lib
    lib = _lib.load()
    lib.b2h_last_error.restype = C.c_char_p
    return lib


def _create(lib, src, dim, autodiff):
    h = C.c_void_p()
    rc = lib.b2h_user_model_create_warp(src.encode(), C.c_int32(dim), C.c_int32(autodiff), C.byref(h))
    msg = lib.b2h_last_error().decode()
    if "libnvrtc" in msg:
        pytest.skip("NVRTC is not installed on this machine")
    return rc, msg


@pytest.mark.parametrize("dim", [1, 65, 1000, 4096])
@pytest.mark.parametrize("name", sorted(warp_sources.AUTODIFF))
def test_warp_reverse_sources_compile(lib, name, dim):
    rc, msg = _create(lib, warp_sources.AUTODIFF[name], dim, 1)
    assert rc != 0 and "loading" in msg, msg


@pytest.mark.parametrize("dim", [0, 1, 65, 1000, 4096])
@pytest.mark.parametrize("name", sorted(warp_sources.HAND))
def test_warp_hand_written_sources_compile(lib, name, dim):
    rc, msg = _create(lib, warp_sources.HAND[name], dim, 0)
    assert rc != 0 and "loading" in msg, msg


@pytest.mark.parametrize("autodiff", [0, 1])
def test_warp_compile_error_reports_the_log(lib, autodiff):
    src = ("template <typename S, typename T> __device__ S log_density(const S* q, int d, const T* data, const Warp& w) "
           "{ return undefined_symbol; }") if autodiff else \
          ("template <typename T> __device__ T potential_and_grad(const T* q, T* g, int d, const T* data, const Warp& w) "
           "{ return undefined_symbol; }")
    rc, msg = _create(lib, src, 70, autodiff)
    assert rc != 0 and "does not compile" in msg and "undefined_symbol" in msg, msg


@pytest.mark.parametrize("dim", [0, -1, 4097])
def test_warp_reverse_dim_is_checked(lib, dim):
    rc, msg = _create(lib, warp_sources.FUNNEL_WARP, dim, 1)
    assert rc != 0 and "dim must be" in msg, msg


def test_warp_autodiff_flag_is_checked(lib):
    rc, msg = _create(lib, warp_sources.FUNNEL_WARP, 10, 2)
    assert rc != 0 and "autodiff" in msg, msg


@pytest.mark.parametrize("src,autodiff", [(BANANA_SRC, 0), (FUNNEL_DENSITY, 1)], ids=["hand-written", "autodiff"])
def test_thread_form_source_is_refused(lib, src, autodiff):
    """A source in the thread calling convention must not run with the warp convention."""
    rc, msg = _create(lib, src, 70, autodiff)
    assert rc != 0 and "does not compile" in msg, msg
