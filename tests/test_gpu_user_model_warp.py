"""Warp-per-chain user densities (UserModel(..., warp=True), b2h_user_model_create_warp): the hand-written form against
its NumPy counterpart with guard bands, exact integer cases, warp reverse mode against thread reverse mode and the
hand-written gradient, a collective used nonlinearly, lanes with different operation counts between collectives,
determinism, tape overflow, and NUTS / HMC / window-adaptation parity against the oracle under injected draws."""
import ctypes as C

import numpy as np
import pytest

import parity
from oracle import models as o_models
from test_gpu_user_model_reverse import _raw_call, _ws_bytes, funnel_terms, logistic_data, logistic_terms, rev_model
from warp_sources import (BRANCHY_WARP, FUNNEL_WARP, FUNNEL_WARP_HAND, IID_WARP, LOGISTIC_WARP, QUAD_COLS, QUAD_ROWS,
                          SHARED_WARP, STUDENT_T_WARP)
from test_gpu_user_model import FUNNEL_DENSITY, LOGISTIC_DENSITY

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

U64, U32 = 2.0 ** -53, 2.0 ** -24
BUTTERFLY = 5               # additions a w.sum puts on each path


@pytest.fixture(scope="module")
def ab(cuda_device):
    import aehmc_b200
    return aehmc_b200


def _np(t):
    return t.detach().double().cpu().numpy()


def _dt(dtype):
    return (torch.float64, U64) if dtype == "f64" else (torch.float32, U32)


def warp_model(ab, src, dim, **kw):
    m = ab.models.UserModel(src, dim, warp=True, **kw)
    assert m.warp
    return m


def funnel_host(q):
    return o_models.NealFunnel(q.shape[0]).potential_and_grad(np.asarray(q, dtype=np.float64))


def funnel_u_terms(q):
    return np.abs(q[:, 0]) ** 2 / 18 + np.sum(0.5 * q[:, 1:] ** 2 * np.exp(-q[:, :1]), axis=1) + \
        0.5 * (q.shape[1] - 1) * np.abs(q[:, 0])


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [1, 2, 31, 32, 33, 1000])
def test_hand_written_against_host(ab, d, dtype):
    """The hand-written warp funnel against NumPy at C = 1, 3 and 129 (a partial last block of 4 chains), with NaN
    rows around q and sentinel rows around U and g.  Each value is a sum of the terms funnel_terms bounds, each
    formed with a few roundings: within 4 (d + 16) u sum|t_k|."""
    dt, u = _dt(dtype)
    model = warp_model(ab, FUNNEL_WARP_HAND, d, dtype=dt, host_fn=funnel_host)
    assert not model.reverse and _ws_bytes(ab, model, 129) == 0
    rng = np.random.default_rng(d)
    for Cn in (1, 3, 129):
        q = torch.as_tensor(rng.standard_normal((Cn, d)), dtype=dt).cuda()
        qc = _np(q)
        qb = torch.full((Cn + 2, d), float("nan"), dtype=dt, device="cuda")
        qb[1:-1] = q
        Ub = torch.full((Cn + 2,), -7.0, dtype=dt, device="cuda")
        gb = torch.full((Cn + 2, d), -7.0, dtype=dt, device="cuda")
        row = qb.element_size() * d
        assert _raw_call(ab, model, qb.data_ptr() + row, Ub.data_ptr() + qb.element_size(), gb.data_ptr() + row, Cn,
                         0, 0) == 0
        torch.cuda.synchronize()
        assert torch.isnan(qb[[0, -1]]).all() and torch.equal(qb[1:-1], q)
        assert (_np(Ub[[0, -1]]) == -7.0).all() and (_np(gb[[0, -1]]) == -7.0).all()
        ref = [model.host_fn(qc[c]) for c in range(Cn)]
        tol = 4 * (d + 16) * u
        assert (np.abs(_np(gb[1:-1]) - np.stack([r[1] for r in ref])) <= tol * funnel_terms(qc)).all(), Cn
        assert (np.abs(_np(Ub[1:-1]) - np.array([r[0] for r in ref])) <= tol * funnel_u_terms(qc)).all(), Cn
        U, g = model.potential_and_grad(q)
        assert torch.equal(U, Ub[1:-1]) and torch.equal(g, gb[1:-1])


def _quad_case(d):
    rng = np.random.default_rng(d)
    B = rng.integers(-1, 2, size=(d, d))
    A = (B + B.T).astype(np.float64)
    mu = rng.integers(-1, 2, size=d).astype(np.float64)
    return A, mu, rng


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [65, 200, 1000])
@pytest.mark.parametrize("form", ["rows", "cols"])
def test_integer_quadratic_form_exact(ab, form, d, dtype):
    """Integer A, mu and q, every partial sum an integer or half-integer far below 2^24: U and the gradient A (q - mu)
    are exact in both precisions.  "rows" gives each lane whole rows (every lane touches every input, so the lanes'
    adjoints meet on one input in the same sweep step); "cols" splits each row's coordinates over the lanes (one
    collective per row)."""
    dt, _ = _dt(dtype)
    A, mu, rng = _quad_case(d)
    q = rng.integers(-1, 2, size=(5 if d == 1000 else 9, d)).astype(np.float64)
    model = warp_model(ab, QUAD_ROWS if form == "rows" else QUAD_COLS, d, data=np.concatenate([mu, A.ravel()]),
                       dtype=dt, autodiff=True)
    assert model.reverse
    U, g = model.potential_and_grad(q)
    r = q - mu
    assert np.array_equal(_np(g), r @ A)
    assert np.array_equal(_np(U), 0.5 * np.einsum("ci,ij,cj->c", r, A, r))


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [1, 40, 70])
def test_shared_operand_counts_twice(ab, d, dtype):
    """q[i] * q[i] (an input) and y * y (a node) with both operands the same."""
    dt, _ = _dt(dtype)
    q = np.random.default_rng(3).integers(-50, 50, size=(40, d)).astype(np.float64)
    U, g = warp_model(ab, SHARED_WARP, d, dtype=dt, autodiff=True).potential_and_grad(q)
    assert np.array_equal(_np(g), 20 * q + 6)
    assert np.array_equal(_np(U), np.sum(q * q + (3 * q + 1) ** 2, axis=1))


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [65, 1000])
def test_funnel_warp_against_thread_reverse_and_hand_written(ab, d, dtype):
    """Every lane reuses q[0].  Warp reverse, thread reverse and the hand-written warp gradient are sums of the same
    terms in different orders: within 2 m u sum|t_k|, m = d + 16 enlarged by the butterfly depth."""
    dt, u = _dt(dtype)
    rng = np.random.default_rng(20 + d)
    q = torch.as_tensor(rng.standard_normal((70, d)), dtype=dt).cuda()
    qc = _np(q)
    Uw, gw = warp_model(ab, FUNNEL_WARP, d, dtype=dt, autodiff=True).potential_and_grad(q)
    Ut, gt = rev_model(ab, FUNNEL_DENSITY, d, dtype=dt).potential_and_grad(q)
    Uh, gh = warp_model(ab, FUNNEL_WARP_HAND, d, dtype=dt).potential_and_grad(q)
    m = d + 16 + BUTTERFLY
    S, Su = funnel_terms(qc), funnel_u_terms(qc)
    for g, U in ((gt, Ut), (gh, Uh)):
        err = np.abs(_np(gw) - _np(g))
        assert (err <= 2 * m * u * S).all(), (err / (2 * m * u * S)).max()
        assert (np.abs(_np(Uw) - _np(U)) <= 2 * m * u * Su).all()


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [65, 300])
def test_logistic_warp_against_thread_reverse(ab, d, dtype):
    """Data rows split over the lanes, so every lane reads every beta: within 2 m u sum|t_k|, m = n + d + 16 + 5."""
    dt, u = _dt(dtype)
    rng = np.random.default_rng(30 + d)
    n = 70
    X, y, data = logistic_data(rng, n, d)
    q = torch.as_tensor(0.5 * rng.standard_normal((40, d)), dtype=dt).cuda()
    Uw, gw = warp_model(ab, LOGISTIC_WARP, d, data=data, dtype=dt, autodiff=True).potential_and_grad(q)
    Ut, gt = rev_model(ab, LOGISTIC_DENSITY, d, data=data, dtype=dt).potential_and_grad(q)
    m = n + d + 16 + BUTTERFLY
    tol = 2 * m * u * logistic_terms(_np(q), X, y)
    err = np.abs(_np(gw) - _np(gt))
    assert (err <= tol).all(), (err / tol).max()
    np.testing.assert_allclose(_np(Uw), _np(Ut), rtol=4 * m * u)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [33, 1000])
def test_collective_used_nonlinearly(ab, d, dtype):
    """Student-t, lp = -(nu + d) / 2 log1p(w.sum(q_i^2) / nu), against the analytic gradient (nu + d) q / (nu + |q|^2).
    An adjoint seeded on every lane would scale it by 32; collective adjoints not summed across lanes would drop all
    but one lane's share."""
    dt, u = _dt(dtype)
    nu = 5.0
    rng = np.random.default_rng(40 + d)
    q = torch.as_tensor(rng.standard_normal((37, d)), dtype=dt).cuda()
    qc = _np(q)
    U, g = warp_model(ab, STUDENT_T_WARP, d, data=[nu], dtype=dt, autodiff=True).potential_and_grad(q)
    s = np.sum(qc * qc, axis=1, keepdims=True)
    rtol = 8 * (d + 40) * u
    np.testing.assert_allclose(_np(g), (nu + d) * qc / (nu + s), rtol=rtol, atol=0)
    np.testing.assert_allclose(_np(U), 0.5 * (nu + d) * np.log1p(s[:, 0] / nu), rtol=rtol)


def branchy_host(q):
    q = np.asarray(q, dtype=np.float64)
    d = q.shape[0]
    n = int(abs(q[0]) * 4.0)
    U, g = 0.5 * q[0] * q[0], np.zeros(d)
    g[0] = q[0]
    for k in range(1, n + 1):
        i = 1 + k % (d - 1)
        r = q[i] - 0.1 * k
        U += r * r * (0.5 / k)
        g[i] += r / k
    pos = q > 0
    U += np.sum(0.25 * q[pos] ** 2)
    g[pos] += 0.5 * q[pos]
    return U, g


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_lanes_with_different_op_counts(ab, dtype):
    """d = 37 (not a multiple of 32), a term count that differs between chains (0 to 48 terms, spread over the
    lanes, several lanes on one input), then a branch on each lane's own values between the two collectives."""
    dt, u = _dt(dtype)
    d, Cn = 37, 33
    rng = np.random.default_rng(4)
    q = rng.standard_normal((Cn, d))
    q[:, 0] = np.linspace(-12.0, 12.0, Cn)
    q = _np(torch.as_tensor(q, dtype=dt))
    model = warp_model(ab, BRANCHY_WARP, d, dtype=dt, autodiff=True, tape_nodes=400, host_fn=branchy_host)
    U, g = model.potential_and_grad(q)
    ref = [branchy_host(q[c]) for c in range(Cn)]
    rtol = 1e-13 if dtype == "f64" else 2e-5
    np.testing.assert_allclose(_np(U), [r[0] for r in ref], rtol=rtol)
    np.testing.assert_allclose(_np(g), np.stack([r[1] for r in ref]), rtol=rtol, atol=100 * u)


@pytest.mark.parametrize("density", ["funnel", "logistic"])
def test_determinism(ab, density):
    """Two calls, a chain alone, in a batch of 5, at position 4096 of 4097, and a workspace of 0xFF bytes: bit-identical
    U and g."""
    d = 1000 if density == "funnel" else 100
    rng = np.random.default_rng(50)
    if density == "funnel":
        model = warp_model(ab, FUNNEL_WARP, d, autodiff=True)
    else:
        model = warp_model(ab, LOGISTIC_WARP, d, data=logistic_data(rng, 70, d)[2], autodiff=True)
    q = torch.as_tensor(0.7 * rng.standard_normal((4097, d))).cuda()
    U0, g0 = model.potential_and_grad(q)
    U1, g1 = model.potential_and_grad(q)
    assert torch.equal(U0, U1) and torch.equal(g0, g1)
    for idx in ([4096], [3, 4096, 0, 77, 2048], list(range(1, 4097)) + [0]):
        U, g = model.potential_and_grad(q[idx])
        assert torch.equal(U, U0[idx]) and torch.equal(g, g0[idx]), idx[:5]
    Cn = 7
    nbytes = _ws_bytes(ab, model, Cn)
    ws = torch.full((nbytes,), 255, dtype=torch.uint8, device="cuda")
    U = torch.empty(Cn, dtype=torch.float64, device="cuda")
    g = torch.empty((Cn, d), dtype=torch.float64, device="cuda")
    qs = q[4090:].contiguous()
    assert _raw_call(ab, model, qs.data_ptr(), U.data_ptr(), g.data_ptr(), Cn, ws.data_ptr(), nbytes) == 0
    model.check_tape()
    assert torch.equal(U, U0[4090:]) and torch.equal(g, g0[4090:])


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_workspace_size(ab, dtype):
    """The documented size formula, and one byte less."""
    dt, _ = _dt(dtype)
    es = 8 if dtype == "f64" else 4
    d, Cn = 80, 45
    model = warp_model(ab, FUNNEL_WARP, d, dtype=dt, autodiff=True)
    N, pitch = model.tape_nodes, 32 * Cn
    R = lambda x: (x + 255) // 256 * 256
    want = 256 + 2 * R(N * pitch * 4) + 2 * R(N * pitch * es) + R(N * pitch * es) + R(Cn * d * 2 * es)
    assert _ws_bytes(ab, model, Cn) == want
    q = torch.as_tensor(np.random.default_rng(5).standard_normal((Cn, d)), dtype=dt).cuda()
    U, g = torch.empty(Cn, dtype=dt, device="cuda"), torch.empty_like(q)
    ws = torch.empty(want + 512, dtype=torch.uint8, device="cuda")
    U0, g0 = model.potential_and_grad(q)
    assert _raw_call(ab, model, q.data_ptr(), U.data_ptr(), g.data_ptr(), Cn, ws.data_ptr() + 8, want) == 0
    assert torch.equal(U, U0) and torch.equal(g, g0)
    assert _raw_call(ab, model, q.data_ptr(), U.data_ptr(), g.data_ptr(), Cn, ws.data_ptr(), want - 1) == -4


def test_tape_overflow(ab):
    """A capacity one node short for lane 1 of chain 0 only: that chain gets U = +inf and g = 0, the others are
    unaffected, and check_tape raises with the per-lane count."""
    from aehmc_b200._lib import B200HMCError
    d = 37
    q = np.full((6, d), -0.5)
    q[:, 0] = 1.0
    # chain 0: 34 terms, two of them on lane 1 (k = 2, 34), and a positive q[1] that adds lane 1's only b term; lane 0
    # has two terms and the prior but no b term (q[0] < 0).  Lane 1 needs 12 nodes, no other lane of any chain 11.
    q[0, 0] = -8.5
    q[0, 1] = 1.0
    big = warp_model(ab, BRANCHY_WARP, d, autodiff=True, tape_nodes=1000)
    U0, g0 = big._evaluate(q)
    need = big._tape_needed()
    big._evaluate(q[1:])
    assert 0 < big._tape_needed() < need
    short = warp_model(ab, BRANCHY_WARP, d, autodiff=True, tape_nodes=need - 1)
    with pytest.raises(B200HMCError, match=f"a lane of a chain needed {need} tape nodes, the capacity is {need - 1}"):
        short.potential_and_grad(q)
    U, g = short._evaluate(q)
    assert short._tape_needed() == need
    assert torch.isinf(U[0]) and U[0] > 0 and not g[0].any()
    assert torch.equal(U[1:], U0[1:]) and torch.equal(g[1:], g0[1:])
    exact = warp_model(ab, BRANCHY_WARP, d, autodiff=True, tape_nodes=need)
    U1, g1 = exact.potential_and_grad(q)
    assert torch.equal(U1, U0) and torch.equal(g1, g0)


def test_probed_tape_counts_nodes_per_lane(ab):
    """The funnel at d = 1000: lane 0 holds 32 of the 999 coordinates, 6 nodes each, plus exp(-v) (2 nodes), the
    collective, the prior (3) and the final sum; in the thread form one chain records 5 + 6 (d - 1)."""
    d = 1000
    m = warp_model(ab, FUNNEL_WARP, d, autodiff=True)
    per_lane = -(-(d - 1) // 32)
    assert m.tape_nodes == 2 + 6 * per_lane + 5
    assert rev_model(ab, FUNNEL_DENSITY, d).tape_nodes == 5 + 6 * (d - 1)
    with pytest.raises(ValueError):
        ab.models.UserModel(FUNNEL_WARP_HAND, d, warp=True, tape_nodes=100)


@pytest.mark.parametrize("src,autodiff", [(FUNNEL_WARP_HAND, False), (FUNNEL_WARP, True)],
                         ids=["hand-written", "reverse"])
def test_nuts_parity_funnel(ab, src, autodiff):
    """Tree depth, leapfrog count and divergence flags exact, positions and acceptance within 1e-9 of the oracle."""
    from aehmc_b200 import _engine
    d = 100
    rng = np.random.default_rng(d)
    Cn, T, eps = 12, 2, 0.2
    q0 = rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    ref = parity.oracle_nuts(o_models.NealFunnel(d), q0, eps, np.ones(d), draws, T)
    model = warp_model(ab, src, d, autodiff=autodiff)
    srng = ab.InjectedDraws(draws["z"], draws["u_dir"], draws["u_biased"], draws["u_uniform"])
    info, extras = _engine.run("nuts", model, np.ones(d), srng, ab.nuts.new_state(q0, model), eps, n_transitions=T)
    assert np.array_equal(info.num_doublings.cpu().numpy(), ref["num_doublings"])
    assert np.array_equal(extras["n_leapfrog"].cpu().numpy(), ref["n_leapfrog"])
    assert np.array_equal(info.is_diverging.cpu().numpy().astype(bool), ref["is_diverging"].astype(bool))
    np.testing.assert_allclose(info.state.position.cpu().numpy(), ref["q"], rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(info.acceptance_probability.cpu().numpy(), ref["acceptance_probability"], rtol=1e-9,
                               atol=1e-12)


@pytest.mark.parametrize("src,autodiff", [(FUNNEL_WARP_HAND, False), (FUNNEL_WARP, True)],
                         ids=["hand-written", "reverse"])
def test_hmc_parity_funnel(ab, src, autodiff):
    """One HMC transition of 5 leapfrog steps against the oracle: flags exact, positions within 1e-9."""
    from aehmc_b200 import _engine
    d, Cn, L, eps = 100, 12, 5, 0.1
    rng = np.random.default_rng(7)
    q0 = rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, 1, d)
    ref = parity.oracle_hmc(o_models.NealFunnel(d), q0, eps, np.ones(d), draws, 1, L)
    model = warp_model(ab, src, d, autodiff=autodiff)
    srng = ab.InjectedDraws(z=draws["z"], u_accept=draws["u_accept"])
    info, extras = _engine.run("hmc", model, np.ones(d), srng, ab.hmc.new_state(q0, model), eps, n_transitions=1,
                               num_integration_steps=L)
    assert np.array_equal(info.is_diverging.cpu().numpy().astype(bool), ref["is_diverging"].astype(bool))
    np.testing.assert_allclose(info.state.position.cpu().numpy(), ref["q"], rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(info.acceptance_probability.cpu().numpy(), ref["acceptance_probability"], rtol=1e-9,
                               atol=1e-12)


def test_window_adaptation_warp(ab):
    """A few warm-up steps in the split engine against the oracle's schedule (as test_window_adaptation_reverse)."""
    rng = np.random.default_rng(23)
    Cn, W, d = 6, 12, 80
    mu, sigma = rng.standard_normal(d), np.exp(0.5 * rng.standard_normal(d))
    o_model = o_models.IIDGaussian(mu, sigma)
    model = warp_model(ab, IID_WARP, d, data=np.concatenate([mu, 1.0 / sigma ** 2]), autodiff=True)
    q0 = 0.5 * rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, W, d)
    ref = parity.oracle_nuts(o_model, q0, 1.0, np.ones(d), draws, W, schedule_steps=W)
    srng = ab.InjectedDraws(**{k: draws[k] for k in ("z", "u_dir", "u_biased", "u_uniform")})
    kernel = ab.nuts.new_kernel(srng, model)
    state, (step_size, imm_out), _ = ab.window_adaptation.run(kernel, ab.nuts.new_state(q0, model), W)
    np.testing.assert_allclose(_np(step_size), ref["eps"], rtol=1e-6)
    np.testing.assert_allclose(_np(imm_out), ref["imm"], rtol=1e-6)
    np.testing.assert_allclose(_np(state.position), ref["q"], rtol=1e-5, atol=1e-8)
