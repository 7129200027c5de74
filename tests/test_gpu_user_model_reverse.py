"""Reverse-mode automatic differentiation of user log-densities (b2h_user_model_create_rev): the tape against forward
mode on the same source, exact integer cases, analytic gradients at large dims, control flow that differs between the
chains of a warp, the workspace guards, tape overflow, and NUTS parity against the oracle under injected draws."""
import ctypes as C

import numpy as np
import pytest

import parity
from oracle import models as o_models
from test_gpu_user_model import FUNNEL_DENSITY, LOGISTIC_DENSITY

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

U64, U32 = 2.0 ** -53, 2.0 ** -24


@pytest.fixture(scope="module")
def ab(cuda_device):
    import aehmc_b200
    return aehmc_b200


def _np(t):
    return t.detach().double().cpu().numpy()


def rev_model(ab, src, dim, **kw):
    """A reverse-mode UserModel at any dim (the public class picks reverse mode only above dim 64)."""
    class Reverse(ab.models.UserModel):
        FORWARD_MAX_DIM = 0
    m = Reverse(src, dim, autodiff=True, **kw)
    assert m.reverse
    return m


def funnel_terms(q):
    """|terms| whose sum each gradient element of the funnel density is: S[c, i]."""
    v, x = q[:, :1], q[:, 1:]
    S = np.empty_like(q)
    S[:, :1] = np.abs(v) / 9 + np.sum(0.5 * x * x * np.exp(-v), axis=1, keepdims=True) + 0.5 * x.shape[1]
    S[:, 1:] = np.abs(x) * np.exp(-v)
    return S


def logistic_terms(q, X, y):
    s = q @ X.T
    r = np.abs(0.5 * (1 + np.tanh(0.5 * s)) - y)
    return np.abs(q) + r @ np.abs(X)


def logistic_data(rng, n, d):
    X = rng.standard_normal((n, d)) / np.sqrt(d)
    y = (rng.random(n) < 0.5).astype(np.float64)
    return X, y, np.concatenate([[n], X.ravel(), y])


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [1, 2, 7, 33, 64])
def test_forward_and_reverse_agree(ab, d, dtype):
    """Same source, both modes.  Every value is computed by the same expression, so U is bit-identical.  Each gradient
    element is a sum of the same chain-rule terms t_k in both modes, formed from identical partials; the modes differ
    only in the order of the adjoint sums and the association of each term's product.  With m the number of
    operations on the longest path (m <= number of terms + depth), each mode's gradient lies within gamma_m * sum|t_k|
    of the exact sum of the computed terms, so |g_fwd - g_rev| <= 2 m u sum|t_k|, u the unit roundoff."""
    dt, u = (torch.float64, U64) if dtype == "f64" else (torch.float32, U32)
    rng = np.random.default_rng(d)
    q = rng.standard_normal((70, d))
    qd = torch.as_tensor(q, dtype=dt).cuda()
    q_cast = _np(qd)
    n = 20
    X, y, data = logistic_data(rng, n, d)
    for src, kw, S, m in ((FUNNEL_DENSITY, {}, funnel_terms(q_cast), d + 16),
                          (LOGISTIC_DENSITY, {"data": data}, logistic_terms(q_cast, X, y), n + d + 16)):
        fwd = ab.models.UserModel(src, d, dtype=dt, autodiff=True, **kw)
        rev = rev_model(ab, src, d, dtype=dt, **kw)
        assert not fwd.reverse
        Uf, gf = fwd.potential_and_grad(qd)
        Ur, gr = rev.potential_and_grad(qd)
        assert torch.equal(Uf, Ur)
        err = np.abs(_np(gf) - _np(gr))
        tol = 2 * m * u * S
        assert (err <= tol).all(), (err / tol).max()


QUAD = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data) {
    // -1/2 (q - mu)^T A (q - mu); data = [mu (d), A (d x d)]
    const T* mu = data;
    const T* A = data + d;
    S lp = (T)0;
    for (int i = 0; i < d; ++i) {
        S t = (T)0;
        for (int j = 0; j < d; ++j) t += (q[j] - mu[j]) * A[i * d + j];
        lp -= (T)0.5 * ((q[i] - mu[i]) * t);
    }
    return lp;
}
"""


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("d", [65, 200])
def test_integer_quadratic_form_exact(ab, d, dtype):
    """Integer A (symmetric), mu and q: every partial sum is an integer or half-integer far below 2^24, so U and the
    gradient A (q - mu) are exact in both precisions."""
    dt = torch.float64 if dtype == "f64" else torch.float32
    rng = np.random.default_rng(d)
    B = rng.integers(-2, 3, size=(d, d))
    A = (B + B.T).astype(np.float64)
    mu = rng.integers(-2, 3, size=d).astype(np.float64)
    q = rng.integers(-3, 4, size=(9, d)).astype(np.float64)
    model = ab.models.UserModel(QUAD, d, data=np.concatenate([mu, A.ravel()]), dtype=dt, autodiff=True)
    assert model.reverse
    U, g = model.potential_and_grad(q)
    r = q - mu
    assert np.array_equal(_np(g), r @ A)
    assert np.array_equal(_np(U), 0.5 * np.einsum("ci,ij,cj->c", r, A, r))


SHARED = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data) {
    S lp = (T)0;
    for (int i = 0; i < d; ++i) {
        const S y = (T)3 * q[i] + (T)1;     // one node (the + 1 aliases it)
        lp -= q[i] * q[i] + y * y;          // both operands of each product are the same node
    }
    return lp;
}
"""


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_shared_operand_counts_twice(ab, dtype):
    dt = torch.float64 if dtype == "f64" else torch.float32
    d = 70
    q = np.random.default_rng(3).integers(-50, 50, size=(40, d)).astype(np.float64)
    U, g = ab.models.UserModel(SHARED, d, dtype=dt, autodiff=True).potential_and_grad(q)
    assert np.array_equal(_np(g), 20 * q + 6)
    assert np.array_equal(_np(U), np.sum(q * q + (3 * q + 1) ** 2, axis=1))


def test_funnel_d1000_matches_builtin(ab):
    """Both gradients are the same sums of terms (the built-in kernel's own order): within 2 (d + 16) u sum|t_k|."""
    d = 1000
    rng = np.random.default_rng(11)
    q = rng.standard_normal((64, d))
    q[:, 0] = 2 * rng.standard_normal(64)
    model = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True)
    assert model.reverse and model.tape_nodes == 5 + 6 * (d - 1)
    U, g = model.potential_and_grad(q)
    U0, g0 = ab.models.NealFunnel(d).potential_and_grad(q)
    S = funnel_terms(q)
    assert (np.abs(_np(g) - _np(g0)) <= 2 * (d + 16) * U64 * S).all()
    Us = np.abs(q[:, 0]) ** 2 / 18 + np.sum(0.5 * q[:, 1:] ** 2 * np.exp(-q[:, :1]), axis=1) + 0.5 * (d - 1) * np.abs(q[:, 0])
    assert (np.abs(_np(U) - _np(U0)) <= 2 * (d + 16) * U64 * Us).all()


@pytest.mark.parametrize("d", [128, 300])
def test_logistic_matches_oracle(ab, d):
    """Against the oracle's NumPy model.  Besides the summation order (2 m u sum|t_k|, m = n + d + 16), each s_i = x_i . q
    carries an error up to d u sum_j |x_ij q_j| that moves the residual by at most a quarter of it."""
    rng = np.random.default_rng(d)
    n = 64
    X, y, data = logistic_data(rng, n, d)
    q = 0.5 * rng.standard_normal((8, d))
    model = ab.models.UserModel(LOGISTIC_DENSITY, d, data=data, autodiff=True)
    U, g = model.potential_and_grad(q)
    om = o_models.LogisticRegression(X, y, 1.0)
    ref = [om.potential_and_grad(q[c]) for c in range(q.shape[0])]
    m = n + d + 16
    ds = d * U64 * (np.abs(q) @ np.abs(X).T)              # [C, n] bound on the error of s
    tol_g = 2 * m * U64 * logistic_terms(q, X, y) + 0.25 * ds @ np.abs(X)
    assert (np.abs(_np(g) - np.stack([r[1] for r in ref])) <= tol_g).all()
    s = q @ X.T
    sp = np.maximum(s, 0) + np.log1p(np.exp(-np.abs(s)))
    tol_u = 2 * m * U64 * (np.sum(sp + np.abs(s * y), axis=1) + 0.5 * np.sum(q * q, axis=1)) + np.sum(ds, axis=1)
    assert (np.abs(_np(U) - np.array([r[0] for r in ref])) <= tol_u).all()


BRANCHY = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data) {
    // the number of terms depends on the chain's own q[0]
    const int n = (int)(fabs(q[0].v) * (T)4);
    S lp = (T)(-0.5) * square(q[0]);
    for (int k = 1; k <= n; ++k) {
        const int i = 1 + k % (d - 1);
        lp -= square(q[i] - (T)(0.1 * k)) * (T)(0.5 / k);
    }
    return lp;
}
"""


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
    return U, g


def test_control_flow_differs_between_chains(ab):
    d, Cn = 70, 33
    rng = np.random.default_rng(4)
    q = rng.standard_normal((Cn, d))
    q[:, 0] = np.linspace(-12.0, 12.0, Cn)             # 0 to 48 loop trips, different in every lane of the warp
    model = ab.models.UserModel(BRANCHY, d, autodiff=True, tape_nodes=400, host_fn=branchy_host)
    U, g = model.potential_and_grad(q)
    ref = [branchy_host(q[c]) for c in range(Cn)]
    np.testing.assert_allclose(_np(U), [r[0] for r in ref], rtol=1e-13)
    np.testing.assert_allclose(_np(g), np.stack([r[1] for r in ref]), rtol=1e-13, atol=1e-15)


def _raw_call(ab, model, q, U, g, Cn, ws, nbytes):
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    m = model.struct()
    return lib.b2h_potential_and_grad(backend.context(model.device), C.byref(m), backend.code(model.dtype),
                                      C.c_void_p(q), C.c_void_p(U), C.c_void_p(g), C.c_int64(Cn), C.c_void_p(ws),
                                      C.c_int64(nbytes))


def _ws_bytes(ab, model, Cn):
    from aehmc_b200 import _lib, backend
    m = model.struct()
    return _lib.load().b2h_potential_workspace_bytes(C.byref(m), backend.code(model.dtype), C.c_int64(Cn))


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_guards_and_workspace(ab, dtype):
    """NaN rows around q, sentinels around U and g, a workspace of 0xFF bytes, the documented size formula and one
    byte less."""
    dt = torch.float64 if dtype == "f64" else torch.float32
    es = 8 if dtype == "f64" else 4
    d, Cn = 80, 45
    model = ab.models.UserModel(FUNNEL_DENSITY, d, dtype=dt, autodiff=True)
    q = torch.as_tensor(np.random.default_rng(5).standard_normal((Cn, d)), dtype=dt).cuda()
    U0, g0 = model.potential_and_grad(q)

    N, pitch = model.tape_nodes, 64
    R = lambda x: (x + 255) // 256 * 256
    want = 256 + 2 * R(N * pitch * 4) + 2 * R(N * pitch * es) + R((d + N) * pitch * es)
    assert _ws_bytes(ab, model, Cn) == want

    qb = torch.full((Cn + 2, d), float("nan"), dtype=dt, device="cuda")
    qb[1:-1] = q
    Ub = torch.full((Cn + 2,), -7.0, dtype=dt, device="cuda")
    gb = torch.full((Cn + 2, d), -7.0, dtype=dt, device="cuda")
    ws = torch.full((want + 512,), 255, dtype=torch.uint8, device="cuda")
    es_q = qb.element_size() * d
    # workspace at an odd offset: the tape aligns itself inside the documented size
    rc = _raw_call(ab, model, qb.data_ptr() + es_q, Ub.data_ptr() + qb.element_size(), gb.data_ptr() + es_q, Cn,
                   ws.data_ptr() + 8, want)
    assert rc == 0
    model.check_tape()
    assert torch.equal(Ub[1:-1], U0) and torch.equal(gb[1:-1], g0)
    assert (_np(Ub[[0, -1]]) == -7.0).all() and (_np(gb[[0, -1]]) == -7.0).all()
    rc = _raw_call(ab, model, q.data_ptr(), Ub.data_ptr(), gb.data_ptr(), Cn, ws.data_ptr(), want - 1)
    assert rc == -4
    rc = _raw_call(ab, model, q.data_ptr(), Ub.data_ptr(), gb.data_ptr(), Cn, 0, 0)
    assert rc == -4


def test_results_do_not_depend_on_chain_count_or_position(ab):
    d, Cmax = 70, 4097
    rng = np.random.default_rng(6)
    q = rng.standard_normal((Cmax, d))
    model = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True)
    U_all, g_all = model.potential_and_grad(q)
    for Cn in (1, 31, 32, 33, 4097):
        idx = (np.arange(Cn) * 7 + Cn) % Cmax          # each chain at another position than in the full call
        U, g = model.potential_and_grad(q[idx])
        assert torch.equal(U, U_all[idx]) and torch.equal(g, g_all[idx]), Cn


def test_tape_overflow(ab):
    from aehmc_b200 import _engine
    from aehmc_b200._lib import B200HMCError
    d = 100
    need = 5 + 6 * (d - 1)
    probed = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True)
    assert probed.tape_nodes == need
    q = np.random.default_rng(8).standard_normal((40, d))
    U0, g0 = probed.potential_and_grad(q)
    exact = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True, tape_nodes=need)
    U1, g1 = exact.potential_and_grad(q)
    assert torch.equal(U1, U0) and torch.equal(g1, g0)

    short = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True, tape_nodes=need - 1)
    with pytest.raises(B200HMCError, match=f"needed {need} tape nodes, the capacity is {need - 1}"):
        short.potential_and_grad(q)
    U, g = short._evaluate(q)           # the policy behind the error: the chain is rejected
    short._tape_needed()
    assert torch.isinf(U).all() and (U > 0).all() and not g.any()
    draws = parity.random_draws(np.random.default_rng(9), 40, 1, d)
    srng = ab.InjectedDraws(draws["z"], draws["u_dir"], draws["u_biased"], draws["u_uniform"])
    with pytest.raises(B200HMCError, match=f"needed {need} tape nodes"):
        _engine.run("nuts", short, np.ones(d), srng, ab.nuts.new_state(q, probed), 0.2, n_transitions=1)

    # the count is read and reset per call: a later call that fits succeeds
    m = ab.models.UserModel(BRANCHY, d, autodiff=True, tape_nodes=20)
    big = np.zeros((3, d)); big[:, 0] = 5.0
    with pytest.raises(B200HMCError, match="needed"):
        m.potential_and_grad(big)
    small = np.zeros((3, d)); small[:, 0] = 0.5
    U, g = m.potential_and_grad(small)
    assert np.isfinite(_np(U)).all()


def test_forward_or_reverse_follows_the_dimension(ab):
    f = ab.models.UserModel(FUNNEL_DENSITY, 64, autodiff=True)
    r = ab.models.UserModel(FUNNEL_DENSITY, 65, autodiff=True)
    assert not f.reverse and f.tape_nodes == 0 and _ws_bytes(ab, f, 100) == 0
    assert r.reverse and r.tape_nodes == 5 + 6 * 64 and _ws_bytes(ab, r, 100) > 0
    with pytest.raises(ValueError):
        ab.models.UserModel(FUNNEL_DENSITY, 64, autodiff=True, tape_nodes=100)


@pytest.mark.parametrize("d,group", [(100, 0), (1000, 256)])
def test_nuts_parity_funnel(ab, d, group):
    """Tree depth, leapfrog count and divergence flags exact, positions and acceptance within 1e-9 of the oracle.
    d = 1000 runs the engine with one CTA per chain."""
    from aehmc_b200 import _engine
    rng = np.random.default_rng(d)
    Cn, T = 12, 2
    q0 = rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    eps = 0.2 if d == 100 else 0.1
    ref = parity.oracle_nuts(o_models.NealFunnel(d), q0, eps, np.ones(d), draws, T)
    model = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True)
    assert model.reverse
    srng = ab.InjectedDraws(draws["z"], draws["u_dir"], draws["u_biased"], draws["u_uniform"])
    info, extras = _engine.run("nuts", model, np.ones(d), srng, ab.nuts.new_state(q0, model), eps, n_transitions=T,
                               group=group)
    assert np.array_equal(info.num_doublings.cpu().numpy(), ref["num_doublings"])
    assert np.array_equal(extras["n_leapfrog"].cpu().numpy(), ref["n_leapfrog"])
    assert np.array_equal(info.is_diverging.cpu().numpy().astype(bool), ref["is_diverging"].astype(bool))
    np.testing.assert_allclose(info.state.position.cpu().numpy(), ref["q"], rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(info.acceptance_probability.cpu().numpy(), ref["acceptance_probability"], rtol=1e-9,
                               atol=1e-12)


def test_window_adaptation_reverse(ab):
    """A few warm-up steps in the split engine against the oracle's schedule (as test_window_adaptation_in_split_mode)."""
    rng = np.random.default_rng(23)
    Cn, W, d = 6, 12, 80
    src = r"""
    template <typename S, typename T>
    __device__ S log_density(const S* q, int d, const T* data) {
        S lp = (T)0;
        for (int i = 0; i < d; ++i) lp -= (T)0.5 * square(q[i] - data[i]) * data[d + i];
        return lp;
    }"""
    mu, sigma = rng.standard_normal(d), np.exp(0.5 * rng.standard_normal(d))
    o_model = o_models.IIDGaussian(mu, sigma)
    model = ab.models.UserModel(src, d, data=np.concatenate([mu, 1.0 / sigma ** 2]), autodiff=True)
    assert model.reverse
    q0 = 0.5 * rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, W, d)
    ref = parity.oracle_nuts(o_model, q0, 1.0, np.ones(d), draws, W, schedule_steps=W)
    srng = ab.InjectedDraws(**{k: draws[k] for k in ("z", "u_dir", "u_biased", "u_uniform")})
    kernel = ab.nuts.new_kernel(srng, model)
    state, (step_size, imm_out), _ = ab.window_adaptation.run(kernel, ab.nuts.new_state(q0, model), W)
    np.testing.assert_allclose(_np(step_size), ref["eps"], rtol=1e-6)
    np.testing.assert_allclose(_np(imm_out), ref["imm"], rtol=1e-6)
    np.testing.assert_allclose(_np(state.position), ref["q"], rtol=1e-5, atol=1e-8)


def test_integrator_and_trajectory_closures(ab):
    """One velocity-Verlet step and one sub-tree through the stand-alone closures, against the built-in funnel."""
    d, Cn, maxd = 90, 20, 5
    rng = np.random.default_rng(12)
    q0 = rng.standard_normal((Cn, d))
    p0 = rng.standard_normal((Cn, d))
    imm = np.exp(0.2 * rng.standard_normal(d))
    rev = ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True)
    ref = ab.models.NealFunnel(d)
    draws = parity.random_draws(rng, Cn, 1, d, maxd)
    dirs = np.where(rng.random(Cn) < 0.5, 1, -1).astype(np.int8)
    out = []
    for model in (rev, ref):
        mg, ke, ut = ab.metrics.gaussian_metric(imm, dtype=model.dtype)
        integ = ab.integrators.velocity_verlet(model, ke)
        U, g = model.potential_and_grad(q0)
        st = ab.integrators.IntegratorState(torch.as_tensor(q0).cuda(), torch.as_tensor(p0).cuda(), U, g)
        step = integ(st, 0.1)
        new_ts, upd, crit = ab.termination.iterative_uturn(ut)
        srng = ab.InjectedDraws(None, draws["u_dir"], draws["u_biased"], draws["u_uniform"], None)
        ti = ab.trajectory.dynamic_integration(srng, integ, ke, upd, crit, 1000.0, expansion=3)
        ts = new_ts(st.position, maxd)
        (prop, last, msum, ts2, length, div, term), _ = ti(st, dirs, ts, 8, 0.15, U + ke(st.momentum))
        out.append((step, prop, last, length, div, term))
    (s_r, pr_r, l_r, n_r, dv_r, t_r), (s_b, pr_b, l_b, n_b, dv_b, t_b) = out
    for a, b in ((s_r.position, s_b.position), (s_r.momentum, s_b.momentum), (s_r.potential_energy_grad, s_b.potential_energy_grad)):
        np.testing.assert_allclose(_np(a), _np(b), rtol=1e-11, atol=1e-12)
    assert torch.equal(n_r, n_b) and torch.equal(dv_r, dv_b) and torch.equal(t_r, t_b)
    np.testing.assert_allclose(_np(pr_r.state.position), _np(pr_b.state.position), rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(_np(l_r.position), _np(l_b.position), rtol=1e-9, atol=1e-11)
