"""GPU parity of the batched L1 primitives against the oracle and the reference's own unit fixtures
(reference tests/test_metrics.py, test_termination.py, test_integrators.py, test_algorithms.py)."""
import numpy as np
import pytest

import parity  # noqa: F401
from oracle import adaptation as o_adapt
from oracle import hamiltonian as o_ham
from oracle import models as o_models
from oracle import tree as o_tree

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ab(cuda_device):
    import aehmc_b200
    return aehmc_b200


def _np(t):
    return t.detach().cpu().numpy()


def _models(ab, rng, d=6, n_data=50):
    mu, sigma = rng.standard_normal(d), np.exp(0.4 * rng.standard_normal(d))
    A = rng.standard_normal((d, d))
    prec = A @ A.T / d + 0.5 * np.eye(d)
    X = np.round(rng.standard_normal((n_data, d)) * 8) / 8
    y = (rng.random(n_data) < 0.5).astype(np.float64)
    return [
        (ab.models.IIDGaussian(mu, sigma, const=0.3), o_models.IIDGaussian(mu, sigma, const=0.3), d),
        (ab.models.CorrelatedGaussian(mu, prec), o_models.CorrelatedGaussian(mu, prec), d),
        (ab.models.NealFunnel(10), o_models.NealFunnel(10), 10),
        (ab.models.EightSchools(), o_models.EightSchools(), 10),
        (ab.models.LogisticRegression(X, y, 2.0), o_models.LogisticRegression(X, y, 2.0), d),
    ]


def test_potential_and_grad_all_models(ab):
    rng = np.random.default_rng(0)
    for gm, om, d in _models(ab, rng):
        q = 0.7 * rng.standard_normal((33, d))
        U, g = gm.potential_and_grad(q)
        ref = [om.potential_and_grad(q[c]) for c in range(q.shape[0])]
        np.testing.assert_allclose(_np(U), [r[0] for r in ref], rtol=1e-12, atol=1e-12, err_msg=type(gm).__name__)
        np.testing.assert_allclose(_np(g), [r[1] for r in ref], rtol=1e-11, atol=1e-12, err_msg=type(gm).__name__)
        np.testing.assert_allclose(_np(gm(q)), [-r[0] for r in ref], rtol=1e-12, atol=1e-12)


def test_potential_and_grad_wide_and_fp32(ab):
    rng = np.random.default_rng(1)
    for d in (100, 1000):
        mu, sigma = rng.standard_normal(d), np.exp(0.4 * rng.standard_normal(d))
        q = rng.standard_normal((17, d))
        om = o_models.IIDGaussian(mu, sigma)
        ref = [om.potential_and_grad(q[c]) for c in range(17)]
        for dt, tol in ((torch.float64, 1e-12), (torch.float32, 2e-5)):
            U, g = ab.models.IIDGaussian(mu, sigma, dtype=dt).potential_and_grad(q)
            np.testing.assert_allclose(_np(U), [r[0] for r in ref], rtol=tol)
            np.testing.assert_allclose(_np(g), [r[1] for r in ref], rtol=tol, atol=tol)


# reference tests/test_metrics.py:31-68
@pytest.mark.parametrize("imm, p, expected", [
    (1.0, [[1.0]], 0.5),
    (np.array([1.0]), [[1.0]], 0.5),
    (np.array([1.0, 1.0]), [[1.0, 1.0]], 1.0),
    (np.array([[1.0, 0], [0, 1.0]]), [[1.0, 1.0]], 1.0),
])
def test_gaussian_metric_kinetic_energy(ab, imm, p, expected):
    _, kinetic_energy, _ = ab.metrics.gaussian_metric(imm)
    K = kinetic_energy(torch.tensor(p, dtype=torch.float64, device="cuda"))
    assert K.shape == (1,) and K.item() == expected


# reference tests/test_metrics.py:71-120
@pytest.mark.parametrize("imm", [1.0, np.ones(2), np.eye(2)])
def test_turning(ab, imm):
    _, _, turning = ab.metrics.gaussian_metric(imm)
    d = 1 if np.ndim(imm) == 0 else 2
    ones = torch.ones((1, d), dtype=torch.float64, device="cuda")
    assert turning(ones, ones, ones).item() is True


def test_fail_wrong_mass_matrix_dimension(ab):     # reference tests/test_metrics.py:123-127
    with pytest.raises(ValueError):
        ab.metrics.gaussian_metric(np.ones((2, 2, 2)))


def test_metric_random_vs_oracle(ab):
    rng = np.random.default_rng(2)
    C, d = 19, 7
    A = rng.standard_normal((d, d))
    dense = A @ A.T / d + 0.3 * np.eye(d)
    pc = np.exp(0.3 * rng.standard_normal((C, d)))
    for imm_g, imm_o in ((0.7, lambda c: np.full(d, 0.7)), (pc[0], lambda c: pc[0]), (dense, lambda c: dense),
                         (ab.metrics.per_chain(pc), lambda c: pc[c])):
        gen, kin, turn = ab.metrics.gaussian_metric(imm_g)
        p, pl, ps = (rng.standard_normal((C, d)) for _ in range(3))
        K = _np(kin(p))
        T = _np(turn(pl, p, ps))
        z = rng.standard_normal((C, 1, d))
        mom = _np(gen(ab.InjectedDraws(z), num_chains=C, dim=d))
        for c in range(C):
            ogen, okin, oturn = o_ham.gaussian_metric(imm_o(c))

            class Z:
                def normal(self, shape, c=c):
                    return z[c, 0]
            assert K[c] == pytest.approx(okin(p[c]), rel=1e-12)
            assert bool(T[c]) == oturn(pl[c], p[c], ps[c])
            np.testing.assert_allclose(mom[c], ogen(Z()), rtol=1e-11, atol=1e-13)


def test_velocity_verlet_all_models_and_metrics(ab):
    """integrators.velocity_verlet one_step / static_integration vs the oracle (1e-10, fp64)."""
    rng = np.random.default_rng(3)
    for gm, om, d in _models(ab, rng):
        C = 9
        A = rng.standard_normal((d, d))
        dense = A @ A.T / d + 0.5 * np.eye(d)
        pc = np.exp(0.2 * rng.standard_normal((C, d)))
        for imm_g, imm_o in ((0.9, lambda c: np.full(d, 0.9)), (pc[0], lambda c: pc[0]),
                             (ab.metrics.per_chain(pc), lambda c: pc[c]), (dense, lambda c: dense)):
            _, kin, _ = ab.metrics.gaussian_metric(imm_g)
            step = ab.integrators.velocity_verlet(gm, kin)
            q0, p0 = 0.5 * rng.standard_normal((C, d)), rng.standard_normal((C, d))
            eps = 0.05 * np.exp(0.2 * rng.standard_normal(C))
            state = ab.integrators.new_integrator_state(gm, q0, torch.tensor(p0, device="cuda"))
            for n_steps in (1, 4):
                out = step(state, torch.tensor(eps), n_steps=n_steps) if n_steps > 1 else step(state, torch.tensor(eps))
                for c in range(C):
                    _, okin, _ = o_ham.gaussian_metric(imm_o(c))
                    ostep = o_ham.velocity_verlet(om.potential_and_grad, okin)
                    s = o_ham.new_integrator_state(om.potential_and_grad, q0[c], p0[c])
                    for _ in range(n_steps):
                        s = ostep(s, eps[c])
                    what = f"{type(gm).__name__} steps={n_steps}"
                    np.testing.assert_allclose(_np(out.position[c]), s.position, rtol=1e-10, atol=1e-12, err_msg=what)
                    np.testing.assert_allclose(_np(out.momentum[c]), s.momentum, rtol=1e-10, atol=1e-12, err_msg=what)
                    np.testing.assert_allclose(_np(out.potential_energy_grad[c]), s.potential_energy_grad, rtol=1e-10, atol=1e-11, err_msg=what)
                    assert out.potential_energy[c].item() == pytest.approx(s.potential_energy, rel=1e-10, abs=1e-12)


def test_velocity_verlet_reference_examples(ab):
    """reference tests/test_integrators.py: harmonic oscillator q=sin(1), p=cos(1) after 100 steps of 0.01,
    energy conserved to 1e-4 (free fall / circular motion need a user potential: oracle only)."""
    model = ab.models.IIDGaussian([0.0], [1.0])
    _, kin, _ = ab.metrics.gaussian_metric(np.array([1.0]))
    step = ab.integrators.velocity_verlet(model, kin)
    integrate = ab.trajectory.static_integration(step, 100)
    s0 = ab.integrators.new_integrator_state(model, np.zeros((1, 1)), torch.ones((1, 1), dtype=torch.float64, device="cuda"))
    s1, _ = integrate(s0, 0.01)
    assert s1.position.item() == pytest.approx(np.sin(1.0), abs=1e-2)
    assert s1.momentum.item() == pytest.approx(np.cos(1.0), abs=1e-2)
    e0 = s0.potential_energy + kin(s0.momentum)
    e1 = s1.potential_energy + kin(s1.momentum)
    assert e1.item() == pytest.approx(e0.item(), rel=1e-4)


def test_vectorised_leapfrog_matches_scalar_path(ab):
    rng = np.random.default_rng(4)
    C = 64
    for d, dt in ((128, torch.float64), (100, torch.float64), (128, torch.float32), (101, torch.float32)):
        mu, sigma = rng.standard_normal(d), np.exp(0.3 * rng.standard_normal(d))
        model = ab.models.IIDGaussian(mu, sigma, dtype=dt)
        om = o_models.IIDGaussian(mu, sigma)
        imm = sigma ** 2
        _, kin, _ = ab.metrics.gaussian_metric(imm, dtype=dt)
        step = ab.integrators.velocity_verlet(model, kin)
        q0, p0 = rng.standard_normal((C, d)), rng.standard_normal((C, d))
        out = step(ab.integrators.new_integrator_state(model, q0, torch.tensor(p0, device="cuda", dtype=dt)), 0.1, n_steps=3)
        _, okin, _ = o_ham.gaussian_metric(imm)
        ostep = o_ham.velocity_verlet(om.potential_and_grad, okin)
        tol = 1e-11 if dt == torch.float64 else 3e-5
        for c in (0, 17, 63):
            s = o_ham.new_integrator_state(om.potential_and_grad, q0[c], p0[c])
            for _ in range(3):
                s = ostep(s, 0.1)
            np.testing.assert_allclose(_np(out.position[c]), s.position, rtol=tol, atol=tol)
            np.testing.assert_allclose(_np(out.momentum[c]), s.momentum, rtol=tol, atol=tol)
            assert out.potential_energy[c].item() == pytest.approx(s.potential_energy, rel=tol * 10)


# reference tests/test_termination.py:12-48
@pytest.mark.parametrize("checkpoint_idxs, expected_turning",
                         [((3, 3), True), ((3, 2), False), ((0, 0), False), ((0, 1), True), ((1, 3), True)])
def test_iterative_turning_termination(ab, checkpoint_idxs, expected_turning):
    _, _, is_turning = ab.metrics.gaussian_metric(np.ones(1))
    _, _, is_iterative_turning = ab.termination.iterative_uturn(is_turning)
    dev = "cuda"
    mck = torch.tensor([1.0, 2.0, 3.0, -2.0], dtype=torch.float64, device=dev).reshape(1, 4, 1)
    sck = torch.tensor([2.0, 4.0, 4.0, -1.0], dtype=torch.float64, device=dev).reshape(1, 4, 1)
    state = ab.termination.TerminationState(mck, sck, torch.tensor([checkpoint_idxs[0]], device=dev),
                                            torch.tensor([checkpoint_idxs[1]], device=dev))
    out = is_iterative_turning(state, torch.tensor([[3.0]], dtype=torch.float64, device=dev),
                               torch.tensor([[1.0]], dtype=torch.float64, device=dev))
    assert out.item() is expected_turning


def test_leaf_idx_to_ckpt_idx(ab):                # reference tests/test_termination.py:51-62
    steps = torch.tensor([0, 6, 7, 13, 15], device="cuda")
    imin, imax = ab.termination._find_storage_indices(steps)
    assert list(zip(_np(imin).tolist(), _np(imax).tolist())) == [(1, 0), (3, 2), (0, 2), (2, 2), (0, 3)]
    steps = torch.arange(1, 3000, device="cuda")
    imin, imax = ab.termination._find_storage_indices(steps)
    ref = [o_tree._find_storage_indices(s) for s in range(1, 3000)]
    assert _np(imin).tolist() == [r[0] for r in ref] and _np(imax).tolist() == [r[1] for r in ref]


@pytest.mark.parametrize("num_dims", [1, 3])
def test_termination_update(ab, num_dims):        # reference tests/test_termination.py:65-91
    _, _, is_turning = ab.metrics.gaussian_metric(np.ones(num_dims))
    new_state, update, _ = ab.termination.iterative_uturn(is_turning)
    ones = torch.ones((2, num_dims), dtype=torch.float64, device="cuda")
    state = new_state(ones, 4)
    update(state, ones, ones, 1)
    odd = update(state, ones, ones, 5)
    assert torch.count_nonzero(odd.momentum_checkpoints) == 0 and torch.count_nonzero(odd.momentum_sum_checkpoints) == 0
    even = update(state, ones, 2 * ones, 6)
    assert _np(even.min_index).tolist() == [3, 3] and _np(even.max_index).tolist() == [2, 2]
    np.testing.assert_array_equal(_np(even.momentum_checkpoints[:, 2]), 2 * np.ones((2, num_dims)))
    zero = update(even, ones, 3 * ones, 0)          # stale indices at step 0 (SURVEY Q2)
    assert _np(zero.min_index).tolist() == [3, 3] and _np(zero.max_index).tolist() == [2, 2]
    np.testing.assert_array_equal(_np(zero.momentum_checkpoints[:, 2]), 3 * np.ones((2, num_dims)))


def test_dual_averaging(ab):                      # reference tests/test_algorithms.py:10-55
    init, update = ab.algorithms.dual_averaging(gamma=0.5)
    state = init(torch.tensor([0.5, 0.5], dtype=torch.float64, device="cuda"))
    oinit, oupdate = o_adapt.dual_averaging(gamma=0.5)
    ostate = oinit(0.5)
    for _ in range(100):
        state = update(2 * (state.iterates - 1), state)
        ostate = oupdate(2 * (ostate.iterates - 1), ostate)
    assert state.iterates_avg[0].item() == pytest.approx(1.0, 1e-2)
    assert state.iterates[0].item() == pytest.approx(1.0, 1e-2)
    assert state.iterates[1].item() == pytest.approx(ostate.iterates, rel=1e-12)
    assert state.iterates_avg[1].item() == pytest.approx(ostate.iterates_avg, rel=1e-12)
    assert state.step[0].item() == 101


@pytest.mark.parametrize("do_compute_covariance", [True, False])
@pytest.mark.parametrize("n_dim", [1, 3])
def test_welford(ab, n_dim, do_compute_covariance):     # reference tests/test_algorithms.py:96-117
    init, update, final = ab.algorithms.welford_covariance(do_compute_covariance)
    state = init(n_dim, 2, device="cuda")
    for i in range(10):
        state = update(i * torch.ones((2, n_dim), dtype=torch.float64, device="cuda"), *state)
    np.testing.assert_allclose(_np(state[0]), 4.5 * np.ones((2, n_dim)))
    cov = _np(final(state[1], state[2]))
    shape = (2, n_dim, n_dim) if do_compute_covariance else (2, n_dim)
    np.testing.assert_allclose(cov, 55.0 / 6.0 * np.ones(shape))


def test_welford_and_mass_matrix_vs_oracle(ab):
    rng = np.random.default_rng(5)
    C, d, n = 3, 4, 25
    xs = rng.standard_normal((n, C, d)) * np.array([1.0, 2.0, 0.5, 3.0])
    for full in (False, True):
        init, update, final = ab.mass_matrix.covariance_adaptation(full)
        imm, wc = init(d, C, device="cuda")
        oinit, oupdate, ofinal = o_adapt.covariance_adaptation(full)
        ostates = [oinit(d)[1] for _ in range(C)]
        for i in range(n):
            wc = update(torch.tensor(xs[i], device="cuda"), wc)
            ostates = [oupdate(xs[i, c], ostates[c]) for c in range(C)]
        got = _np(final(wc))
        for c in range(C):
            np.testing.assert_allclose(got[c], ofinal(ostates[c]), rtol=1e-12, atol=1e-15)


def test_dense_apply(ab):
    import ctypes as C
    from aehmc_b200 import _lib, backend
    rng = np.random.default_rng(6)
    lib = _lib.load()
    for (Cn, d), dt, tol in (((37, 19), torch.float64, 1e-13), ((300, 257), torch.float64, 1e-13),
                             ((260, 1000), torch.float64, 1e-13), ((64, 112), torch.float64, 1e-13),
                             ((129, 96), torch.float64, 1e-13), ((513, 250), torch.float64, 1e-13),
                             ((4096, 1000), torch.float64, 1e-13), ((131072, 128), torch.float64, 1e-13),
                             ((130, 128), torch.float32, 1e-5)):
        a = rng.standard_normal((Cn, d)); m = rng.standard_normal((d, d))
        ta, tm = torch.tensor(a, dtype=dt, device="cuda"), torch.tensor(m, dtype=dt, device="cuda")
        out = torch.empty_like(ta)
        _lib.check(lib.b2h_dense_apply(backend.context(ta.device), backend.code(dt), backend.ptr(ta), backend.ptr(tm),
                                       backend.ptr(out), C.c_int64(Cn), C.c_int64(d)))
        np.testing.assert_allclose(_np(out), a @ m, rtol=tol, atol=tol * d)


def test_philox_fill_statistics_and_determinism(ab):
    import ctypes as C
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    dev = torch.device("cuda:0")
    Cn, T, d, maxd = 64, 4, 50, 10

    def fill(seed, offset):
        z = torch.empty((Cn, T, d), dtype=torch.float64, device=dev)
        ud = torch.empty((Cn, T, maxd), dtype=torch.float64, device=dev)
        ub = torch.empty_like(ud)
        uu = torch.empty((Cn, T, 1023), dtype=torch.float64, device=dev)
        ua = torch.empty((Cn, T), dtype=torch.float64, device=dev)
        _lib.check(lib.b2h_philox_fill(backend.context(dev), C.c_uint64(seed), C.c_uint64(offset), C.c_uint64(0),
                                       C.c_int64(Cn), C.c_int64(T), C.c_int64(d), C.c_int32(maxd), backend.ptr(z),
                                       backend.ptr(ud), backend.ptr(ub), backend.ptr(uu), backend.ptr(ua)))
        return z, ud, ub, uu, ua
    z, ud, ub, uu, ua = fill(7, 0)
    assert abs(z.mean().item()) < 0.03 and abs(z.std().item() - 1) < 0.03
    assert 0 <= uu.min().item() and uu.max().item() < 1 and abs(uu.mean().item() - 0.5) < 0.01
    z2 = fill(7, 0)[0]
    assert torch.equal(z, z2)
    zoff = fill(7, 16)[0]                       # sharding invariance: chain 16 of shard 0 == chain 0 of shard at offset 16
    assert torch.equal(z[16:], zoff[:Cn - 16])
    assert not torch.equal(z, fill(8, 0)[0])
    from scipy import stats
    assert stats.kstest(_np(z).ravel()[:20000], "norm").pvalue > 1e-3
    assert stats.kstest(_np(uu).ravel()[:20000], "uniform").pvalue > 1e-3


def test_device_autocov_and_ess_match_host(ab):
    rng = np.random.default_rng(8)
    T, Cn, d = 300, 20, 3
    x = np.zeros((T, Cn, d))
    for t in range(1, T):
        x[t] = 0.7 * x[t - 1] + rng.standard_normal((Cn, d))
    for dt, tol in ((torch.float64, 1e-10), (torch.float32, 1e-4)):
        dev_stats = ab.diagnostics.sufficient_statistics(torch.tensor(x, dtype=dt, device="cuda"), 60)
        host_stats = ab.diagnostics.sufficient_statistics_numpy(x, 60)
        for k in ("sum_mean", "sum_mean_sq", "sum_acov"):
            np.testing.assert_allclose(dev_stats[k], host_stats[k], rtol=tol, atol=tol)
    e_dev = ab.diagnostics.ess(torch.tensor(x, device="cuda"), 60, method="mean")
    e_host = ab.diagnostics.ess_from_statistics(host_stats)
    np.testing.assert_allclose(e_dev, e_host, rtol=1e-8)
    r = ab.diagnostics.rhat(torch.tensor(x, device="cuda"))
    assert np.all(np.abs(r - 1) < 0.1)
