"""tcgen05 / TMA tensor-core path: the bf16 contraction kernel against an exact reference, and the logistic
regression gradient / NUTS transition it feeds against the FMA exactness-reference path."""
import ctypes as C

import numpy as np
import pytest

import parity
from oracle import models as o_models
from tc_dispatch import tc_plan

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ab(cuda_device):
    import aehmc_b200
    return aehmc_b200


def _tc_gemm(A, B, M, N, K, pieces, piece_rows, nsplit):
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    dev = A.device
    out = torch.full((max(nsplit, 1), M, N), float("nan"), dtype=torch.float32, device=dev)
    _lib.check(lib.b2h_tc_gemm_bf16(backend.context(dev), backend.ptr(A), C.c_int64(A.shape[1]), backend.ptr(B),
                                    C.c_int64(B.shape[1]), backend.ptr(out), C.c_int64(M), C.c_int64(N), C.c_int64(K),
                                    C.c_int32(pieces), C.c_int64(piece_rows), C.c_int64(N), C.c_int32(nsplit),
                                    C.c_int64(M * N)))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("M, N, K, pieces, nsplit", [
    (128, 128, 64, 1, 1), (128, 128, 256, 1, 1), (256, 384, 128, 1, 1), (300, 200, 136, 3, 1),
    (128, 128, 2048, 1, 4), (4096, 128, 1024, 3, 3), (192, 1000, 128, 3, 1),
    (256, 20000, 128, 3, 1), (300, 19000, 64, 1, 1),      # A-resident variant (short K, many column tiles)
])
def test_tc_gemm_matches_exact_reference(ab, M, N, K, pieces, nsplit):
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn((pieces * M, K), device="cuda", generator=g).bfloat16()
    B = torch.randn((N, K), device="cuda", generator=g).bfloat16()
    out = _tc_gemm(A, B, M, N, K, pieces, M, nsplit)
    planes = tc_plan(M, N, K, pieces, nsplit)["planes"]       # the split clamping of the host dispatch
    got = out.double()
    ref = sum(A[p * M:(p + 1) * M].double() @ B.double().T for p in range(pieces))
    assert not torch.isnan(got[:planes]).any(), "a plane the dispatch writes was left unwritten"
    assert torch.isnan(got[planes:]).all(), "a plane beyond the dispatch's count was written"
    total = got[:planes].sum(0)
    scale = (A.double().abs().max() * B.double().abs().max() * K * pieces).item()
    assert (total - ref).abs().max().item() < 2e-6 * scale


def _logistic_case(rng, N, d):
    X = torch.tensor(rng.standard_normal((N, d)), dtype=torch.float32).bfloat16().double().numpy()
    beta = rng.standard_normal(d) / np.sqrt(d)
    y = (rng.random(N) < 1 / (1 + np.exp(-X @ beta))).astype(np.float64)
    return X, y


@pytest.mark.parametrize("tc_mode", [True, "bf16x3", "two_kernel"])
@pytest.mark.parametrize("N, d, Cn", [(512, 64, 40), (2048, 128, 130), (20000, 128, 256), (1000, 96, 300), (40000, 128, 700)])
def test_logistic_gradient_tensor_core_vs_fma(ab, N, d, Cn, tc_mode):
    rng = np.random.default_rng(N + d)
    X, y = _logistic_case(rng, N, d)
    q = 0.3 * rng.standard_normal((Cn, d))
    for dt in (torch.float64, torch.float32):
        ref_model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float64)
        tc_model = ab.models.LogisticRegression(X, y, 1.0, dtype=dt, tensor_core=tc_mode)
        U0, g0 = ref_model.potential_and_grad(q)
        U1, g1 = tc_model.potential_and_grad(q)
        gs = g0.abs().max().item()
        assert (g1.double() - g0).abs().max().item() < 2e-5 * gs
        assert ((U1.double() - U0).abs() / U0.abs()).max().item() < 2e-6
    om = o_models.LogisticRegression(X, y, 1.0)
    Uo, go = om.potential_and_grad(q[0])
    assert abs(U1[0].item() - Uo) / abs(Uo) < 1e-5
    np.testing.assert_allclose(g1[0].double().cpu().numpy(), go, atol=2e-5 * gs)


@pytest.mark.parametrize("tc_mode", [True, "bf16x3"])
def test_nuts_logistic_tensor_core_float32_parity(ab, tc_mode):
    """north star: FP32 bar -- positions within 1e-4 of the oracle per transition, tree shapes equal
    (a near-tie U-turn test may flip in float32: >= 90 % must be identical)."""
    from aehmc_b200 import _engine
    rng = np.random.default_rng(77)
    N, d, Cn, T = 1024, 64, 48, 1
    X, y = _logistic_case(rng, N, d)
    q0 = 0.1 * rng.standard_normal((Cn, d))
    imm = np.full(d, 4.0 / N)
    draws = parity.random_draws(rng, Cn, T, d)
    ref = parity.oracle_nuts(o_models.LogisticRegression(X, y, 1.0), q0, 0.4, imm, draws, T)
    model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float32, tensor_core=tc_mode)
    assert model.tc_flag == (4.0 if tc_mode is True else 2.0)
    srng = ab.InjectedDraws(draws["z"], draws["u_dir"], draws["u_biased"], draws["u_uniform"])
    info, extras = _engine.run("nuts", model, imm, srng, ab.nuts.new_state(q0, model), 0.4, n_transitions=T)
    nd = info.num_doublings.cpu().numpy()
    nl = extras["n_leapfrog"].cpu().numpy()
    same = (nd == ref["num_doublings"]) & (nl == ref["n_leapfrog"])
    assert same.mean() >= 0.9
    q = info.state.position.double().cpu().numpy()
    np.testing.assert_allclose(q[same], ref["q"][same], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("scale_exp", [-10, 6])
def test_logistic_fp16_path_follows_the_data_scale(ab, scale_exp):
    """X * 2^k with beta * 2^-k is the same model: the fp16 pieces' scales are tied to the data scale, so the
    gradient (which scales by 2^k) keeps its accuracy for small and large features."""
    rng = np.random.default_rng(3)
    N, d, Cn = 4096, 128, 64
    X, y = _logistic_case(rng, N, d)
    q = 0.3 * rng.standard_normal((Cn, d))
    k = 2.0 ** scale_exp
    ref_model = ab.models.LogisticRegression(X * k, y, 1e6, dtype=torch.float64)           # flat prior: pure likelihood
    tc_model = ab.models.LogisticRegression(X * k, y, 1e6, dtype=torch.float32, tensor_core=True)
    assert tc_model.tc_flag == 4.0
    U0, g0 = ref_model.potential_and_grad(q / k)
    U1, g1 = tc_model.potential_and_grad(q / k)
    assert (g1.double() - g0).abs().max().item() < 2e-5 * g0.abs().max().item()
    assert ((U1.double() - U0).abs() / U0.abs()).max().item() < 2e-6


def test_logistic_fp16_path_rejects_out_of_range_beta(ab):
    """|beta| beyond what the fp16 pieces can carry (255 for unit-scale data) must not give a silently wrong gradient:
    the state gets U = +inf, which the sampler treats as a divergence."""
    rng = np.random.default_rng(4)
    X, y = _logistic_case(rng, 1024, 64)
    model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float64, tensor_core=True)
    q = 0.1 * rng.standard_normal((8, 64))
    q[3, 5] = 400.0
    U, g = model.potential_and_grad(q)
    assert torch.isinf(U[3]) and U[3] > 0
    assert torch.isfinite(torch.cat([U[:3], U[4:]])).all()


@pytest.mark.parametrize("tc_mode", [True, "bf16x3"])
@pytest.mark.parametrize("N, d, Cn", [(256, 64, 20000), (192, 128, 40000)])
def test_logistic_fused_many_chain_tiles_per_cta(ab, N, d, Cn, tc_mode):
    """Few data tiles, many chain tiles: every CTA walks several (chain tile) segments -- beta reload, G drain and the
    partial-plane bookkeeping at each boundary (the c5 shape has ~7 segments per CTA)."""
    rng = np.random.default_rng(N + Cn)
    X, y = _logistic_case(rng, N, d)
    q = 0.3 * rng.standard_normal((Cn, d))
    ref_model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float64)
    tc_model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float32, tensor_core=tc_mode)
    U0, g0 = ref_model.potential_and_grad(q)
    U1, g1 = tc_model.potential_and_grad(q)
    assert (g1.double() - g0).abs().max().item() < 2e-5 * g0.abs().max().item()
    assert ((U1.double() - U0).abs() / U0.abs()).max().item() < 5e-6


def test_logistic_round_features_option(ab):
    """Arbitrary float features: tensor_core=True refuses them unless round_features=True defines the model on the
    bf16-rounded X, in which case every gradient path sees the same matrix."""
    rng = np.random.default_rng(8)
    X = rng.standard_normal((512, 64))                       # not bf16-representable
    y = (rng.random(512) < 0.5).astype(np.float64)
    with pytest.raises(ValueError):
        ab.models.LogisticRegression(X, y, 1.0, tensor_core=True)
    tc = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float32, tensor_core=True, round_features=True)
    ref = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float64, round_features=True)
    assert tc.tc_flag == 4.0 and torch.equal(tc.X.double(), ref.X)
    q = 0.3 * rng.standard_normal((16, 64))
    (U0, g0), (U1, g1) = ref.potential_and_grad(q), tc.potential_and_grad(q)
    assert (g1.double() - g0).abs().max().item() < 2e-5 * g0.abs().max().item()
    assert ((U1.double() - U0).abs() / U0.abs()).max().item() < 5e-6
