"""Per-chain dense inverse mass matrices (B2H_IMM_DENSE_PER_CHAIN): the batched per-chain mat-vec and the per-chain
factorisation against exact references, the metric primitives and the engine (NUTS / HMC, momentum rider, resume)
against the oracle run chain by chain, bit-for-bit agreement with the per-chain diagonal kind, per-chain dense window
adaptation against the reference's ``is_mass_matrix_full=True`` run per chain, and the error paths."""
import ctypes as C
import io

import numpy as np
import pytest

import parity
from oracle import adaptation as o_adapt
from oracle import hamiltonian as o_ham
from oracle import kernels as o_kernels
from oracle import models as o_models

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ab(cuda_device):
    import aehmc_b200
    return aehmc_b200


def _np(t):
    return None if t is None else t.detach().cpu().numpy()


def _spd(rng, C, d, cond=10.0):
    """C random SPD matrices with eigenvalues log-spaced over [1 / cond, 1] in random orientations."""
    out = np.empty((C, d, d))
    for c in range(C):
        Q, _ = np.linalg.qr(rng.standard_normal((d, d)))
        out[c] = (Q * np.logspace(0, -np.log10(cond), d)) @ Q.T
        out[c] = 0.5 * (out[c] + out[c].T)
    return out


def _corr_case(rng, d):
    mu = rng.standard_normal(d)
    cov = _spd(rng, 1, d, 30.0)[0] * 2.0
    return mu, cov, np.linalg.inv(cov)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the batched per-chain mat-vec, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
GUARD = 64
SENTINEL = 12345.0


def _apply_case(ab, lib, dev, gen, Cn, d, dt, tri, off):
    from aehmc_b200 import _lib, backend
    x = torch.randint(-4, 5, (Cn, d), generator=gen, device=dev).to(torch.float64)
    M = torch.randint(-4, 5, (Cn, d, d), generator=gen, device=dev).to(torch.float64)
    k = torch.arange(d, device=dev)
    if tri == 1:
        zero = k[:, None] > k[None, :]                  # upper: M[k][j] = 0 for k > j
    elif tri == 2:
        zero = k[:, None] < k[None, :]
    else:
        zero = torch.zeros((d, d), dtype=torch.bool, device=dev)
    Mref = M.masked_fill(zero, 0.0)
    ref = (x[:, :, None] * Mref).sum(1)                 # integers: exact in float64 whatever the order
    Mgpu = M.masked_fill(zero, float("nan"))            # the zero half must never reach a result
    # NaN guard bands around in and M, a sentinel-filled output with an extra row; pointers offset by `off` elements
    bin_ = torch.full((2 * GUARD + off + Cn * d,), float("nan"), dtype=dt, device=dev)
    bM = torch.full((2 * GUARD + off + Cn * d * d,), float("nan"), dtype=dt, device=dev)
    bout = torch.full((2 * GUARD + off + (Cn + 1) * d,), SENTINEL, dtype=dt, device=dev)
    s = GUARD + off
    bin_[s:s + Cn * d] = x.reshape(-1).to(dt)
    bM[s:s + Cn * d * d] = Mgpu.reshape(-1).to(dt)
    esz = bin_.element_size()
    _lib.check(lib.b2h_dense_apply_per_chain(backend.context(dev), backend.code(dt), C.c_void_p(bin_.data_ptr() + s * esz),
                                             C.c_void_p(bM.data_ptr() + s * esz), C.c_void_p(bout.data_ptr() + s * esz),
                                             C.c_int64(Cn), C.c_int64(d), C.c_int32(tri)))
    got = bout[s:s + Cn * d].double().reshape(Cn, d)
    what = f"C={Cn} d={d} {dt} tri={tri} off={off}"
    assert torch.equal(got, ref), what
    rest = torch.cat([bout[:s], bout[s + Cn * d:]])
    assert bool((rest == SENTINEL).all()), what + ": write outside the output"


@pytest.mark.parametrize("Cn", [1, 7, 70, 4097])
@pytest.mark.parametrize("d", [1, 2, 3, 5, 8, 16, 17, 31, 32, 33, 64, 100, 127, 128])
def test_dense_apply_per_chain_exact(ab, d, Cn):
    from aehmc_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev)
    gen.manual_seed(1000 * d + Cn)
    for dt in (torch.float64, torch.float32):
        for tri in (0, 1, 2):
            for off in (0, 1):                         # off = 1: every pointer misaligned -> scalar path
                _apply_case(ab, lib, dev, gen, Cn, d, dt, tri, off)


def test_dense_apply_per_chain_rejects_bad_arguments(ab):
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    t = torch.zeros(129 * 129 * 2, dtype=torch.float64, device="cuda")
    ctx = backend.context(t.device)
    for Cn, d, tri in ((0, 4, 0), (2, 0, 0), (2, 129, 0), (2, 4, 3), (2, 4, -1)):
        rc = lib.b2h_dense_apply_per_chain(ctx, _lib.F64, backend.ptr(t), backend.ptr(t), backend.ptr(t),
                                           C.c_int64(Cn), C.c_int64(d), C.c_int32(tri))
        assert rc == -1, (Cn, d, tri)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the per-chain factorisation
# ---------------------------------------------------------------------------------------------------------------------
def _factor(ab, A, dt=torch.float64):
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    a = torch.as_tensor(A, dtype=dt, device="cuda").contiguous()
    Cn, d, _ = a.shape
    imm, sq, ch = (torch.empty_like(a) for _ in range(3))
    info = torch.full((Cn,), -7, dtype=torch.int32, device="cuda")
    _lib.check(lib.b2h_dense_factor_per_chain(backend.context(a.device), backend.code(dt), backend.ptr(a), backend.ptr(imm),
                                              backend.ptr(sq), backend.ptr(ch), backend.ptr(info), C.c_int64(Cn),
                                              C.c_int64(d)))
    return _np(imm), _np(sq), _np(ch), _np(info)


def _gamma(n):
    u = 2.0 ** -53
    return n * u / (1 - n * u)


@pytest.mark.parametrize("d", [1, 2, 5, 33, 64, 128])
def test_factor_per_chain_backward_error(ab, d):
    """FP64 error bounds (Higham, Accuracy and Stability of Numerical Algorithms, Thm 10.3 and 8.5), elementwise,
    with gamma_n = n u / (1 - n u), u = 2^-53, and one more gamma for forming each residual in float64:
      Cholesky:             |L L^T - A|      <= 2 gamma_{d+1} |L| |L^T|
      triangular inverse:   column j of X = L^-1 solves (L + dL_j) x_j = e_j with |dL_j| <= gamma_d |L|, so
                            |L X - I| <= gamma_d |L| |X| and X L - I = X (L X - I) L gives
                            |X L - I| <= gamma_d |X| |L| |X| |L| + gamma_d |X| |L|, checked with a factor 2.
    sqrt_t . chol_t^T = X L.  Condition numbers 1 to 1e8."""
    rng = np.random.default_rng(d)
    conds = [1.0, 1e2, 1e4, 1e6, 1e8]
    A = np.concatenate([_spd(rng, 1, d, c) for c in conds])
    imm, X, LT, info = _factor(ab, A)
    assert (info == 0).all()
    np.testing.assert_array_equal(imm, 0.5 * (A + np.transpose(A, (0, 2, 1))))
    for c in range(len(conds)):
        L, Xc = LT[c].T, X[c]
        assert np.array_equal(np.tril(L), L) and np.array_equal(np.tril(Xc), Xc)
        aL, aX = np.abs(L), np.abs(Xc)
        r1 = np.abs(L @ L.T - imm[c])
        assert (r1 <= 2 * _gamma(d + 1) * (aL @ aL.T) + 1e-300).all(), (conds[c], (r1 / (aL @ aL.T)).max())
        r2 = np.abs(Xc @ L - np.eye(d))
        bound = 2 * _gamma(d) * (aX @ aL @ aX @ aL + aX @ aL)
        assert (r2 <= bound).all(), (conds[c], (r2 / bound).max())


def test_factor_per_chain_fp32_is_fp64_rounded(ab):
    """The factorisation runs in FP64 whatever the dtype: FP32 outputs are the FP64 ones rounded."""
    rng = np.random.default_rng(5)
    A = _spd(rng, 6, 17, 1e3).astype(np.float32).astype(np.float64)
    imm64, sq64, ch64, _ = _factor(ab, A)
    imm32, sq32, ch32, info = _factor(ab, A, torch.float32)
    assert (info == 0).all()
    for a32, a64 in ((imm32, imm64), (sq32, sq64), (ch32, ch64)):
        np.testing.assert_array_equal(a32, a64.astype(np.float32))


def test_factor_per_chain_symmetrises_and_flags_indefinite_chains(ab):
    rng = np.random.default_rng(6)
    Cn, d = 9, 6
    A = _spd(rng, Cn, d, 50.0)
    skew = rng.standard_normal((Cn, d, d))
    asym = A + 0.1 * (skew - np.transpose(skew, (0, 2, 1)))
    imm, sq, ch, info = _factor(ab, asym)
    sym = 0.5 * (asym + np.transpose(asym, (0, 2, 1)))
    np.testing.assert_array_equal(imm, sym)
    imm_s, sq_s, ch_s, _ = _factor(ab, sym)
    np.testing.assert_array_equal(sq, sq_s)
    np.testing.assert_array_equal(ch, ch_s)
    bad = [2, 5, 8]
    B = A.copy()
    B[2][3, 3] = -1.0                                    # a negative pivot at k = 3 at the latest
    B[5] = -B[5]                                         # pivot 0 negative
    B[8][:, :] = 0.0                                     # pivot 0 zero
    _, sq, ch, info = _factor(ab, B)
    assert set(np.nonzero(info)[0].tolist()) == set(bad)
    assert info[5] == 1 and info[8] == 1 and 1 <= info[2] <= 4
    for c in range(Cn):
        if c in bad:
            assert np.isnan(sq[c]).all() and np.isnan(ch[c]).all()
        else:
            assert np.isfinite(sq[c]).all() and np.isfinite(ch[c]).all()
    with pytest.raises(ValueError, match="2, 5, 8"):
        ab.metrics.gaussian_metric(ab.metrics.per_chain(torch.tensor(B, device="cuda")))


# ---------------------------------------------------------------------------------------------------------------------
# 3. the metric primitives
# ---------------------------------------------------------------------------------------------------------------------
def test_metric_primitives_per_chain_dense_vs_oracle(ab):
    rng = np.random.default_rng(7)
    Cn, d = 19, 7
    imms = _spd(rng, Cn, d, 100.0)
    gen, kin, turn = ab.metrics.gaussian_metric(ab.metrics.per_chain(imms))
    p, pl, ps = (rng.standard_normal((Cn, d)) for _ in range(3))
    K = _np(kin(p))
    T = _np(turn(pl, p, ps))
    z = rng.standard_normal((Cn, 1, d))
    mom = _np(gen(ab.InjectedDraws(z)))                  # the chain count comes from the metric
    assert mom.shape == (Cn, d)
    for c in range(Cn):
        ogen, okin, oturn = o_ham.gaussian_metric(imms[c])

        class Z:
            def normal(self, shape, c=c):
                return z[c, 0]
        assert K[c] == pytest.approx(okin(p[c]), rel=1e-12)
        assert bool(T[c]) == oturn(pl[c], p[c], ps[c])
        np.testing.assert_allclose(mom[c], ogen(Z()), rtol=1e-11, atol=1e-13)


def test_leapfrog_per_chain_dense_vs_oracle(ab):
    rng = np.random.default_rng(8)
    Cn, d = 9, 6
    mu, cov, prec = _corr_case(rng, d)
    X = np.round(rng.standard_normal((40, d)) * 8) / 8
    y = (rng.random(40) < 0.5).astype(np.float64)
    imms = _spd(rng, Cn, d, 20.0)
    for gm, om in ((ab.models.CorrelatedGaussian(mu, prec), o_models.CorrelatedGaussian(mu, prec)),
                   (ab.models.IIDGaussian(mu, np.ones(d)), o_models.IIDGaussian(mu, np.ones(d))),
                   (ab.models.LogisticRegression(X, y, 2.0), o_models.LogisticRegression(X, y, 2.0))):
        _, kin, _ = ab.metrics.gaussian_metric(ab.metrics.per_chain(imms))
        step = ab.integrators.velocity_verlet(gm, kin)
        q0, p0 = mu + 0.5 * rng.standard_normal((Cn, d)), rng.standard_normal((Cn, d))
        eps = 0.05 * np.exp(0.2 * rng.standard_normal(Cn))
        state = ab.integrators.new_integrator_state(gm, q0, torch.tensor(p0, device="cuda"))
        out = step(state, torch.tensor(eps), n_steps=3)
        for c in range(Cn):
            _, okin, _ = o_ham.gaussian_metric(imms[c])
            ostep = o_ham.velocity_verlet(om.potential_and_grad, okin)
            s = o_ham.new_integrator_state(om.potential_and_grad, q0[c], p0[c])
            for _ in range(3):
                s = ostep(s, eps[c])
            what = type(gm).__name__
            np.testing.assert_allclose(_np(out.position[c]), s.position, rtol=1e-10, atol=1e-12, err_msg=what)
            np.testing.assert_allclose(_np(out.momentum[c]), s.momentum, rtol=1e-10, atol=1e-12, err_msg=what)
            assert out.potential_energy[c].item() == pytest.approx(s.potential_energy, rel=1e-10, abs=1e-12)


# ---------------------------------------------------------------------------------------------------------------------
# 4. bit-for-bit agreement with the per-chain diagonal kind
# ---------------------------------------------------------------------------------------------------------------------
def _engine_out(info, extras):
    out = dict(q=_np(info.state.position), p=_np(info.state.momentum), U=_np(info.state.potential_energy),
               g=_np(info.state.potential_energy_grad), acceptance_probability=_np(info.acceptance_probability),
               is_diverging=_np(info.is_diverging), n_leapfrog=_np(extras["n_leapfrog"]), draws=_np(extras["draws"]))
    if info.num_doublings is not None:
        out.update(num_doublings=_np(info.num_doublings), is_turning=_np(info.is_turning))
    return out


def _run(ab, kind, model, imm, q0, eps, draws, T, group=0, L=3, div_thr=1000.0):
    from aehmc_b200 import _engine
    eps = torch.as_tensor(np.broadcast_to(eps, (q0.shape[0],)).copy(), dtype=torch.float64)
    if kind == "nuts":
        srng = ab.InjectedDraws(**{k: draws[k] for k in ("z", "u_dir", "u_biased", "u_uniform")})
        info, extras = _engine.run("nuts", model, imm, srng, ab.nuts.new_state(q0, model), eps, n_transitions=T,
                                   store_draws=T, group=group, divergence_threshold=div_thr)
    else:
        srng = ab.InjectedDraws(z=draws["z"], u_accept=draws["u_accept"])
        info, extras = _engine.run("hmc", model, imm, srng, ab.hmc.new_state(q0, model), eps, n_transitions=T,
                                   num_integration_steps=L, store_draws=T, group=group, divergence_threshold=div_thr)
    return _engine_out(info, extras)


@pytest.mark.parametrize("kind", ["nuts", "hmc"])
@pytest.mark.parametrize("d, group", [(6, 8), (33, 32), (33, 256)])
def test_diagonal_stored_densely_matches_diagonal_kind(ab, kind, d, group):
    """Every product with a diagonal matrix of powers of 4 (and with its factors, powers of 2) is an exact scaling,
    and the dense sums only add exact zeros, so the dense per-chain kind must reproduce the per-chain diagonal kind
    bit for bit: imm (p - h g) = imm p - h (imm g) exactly, and sqrt(1 / 4^k) z = 2^-k z = z . L^-1."""
    rng = np.random.default_rng(100 + d + group)
    Cn, T = 70, 3
    mu, cov, prec = _corr_case(rng, d)
    diag = 4.0 ** rng.integers(-2, 3, size=(Cn, d))
    dense = np.zeros((Cn, d, d))
    dense[:, np.arange(d), np.arange(d)] = diag
    q0 = mu + rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    model = ab.models.CorrelatedGaussian(mu, prec)
    a = _run(ab, kind, model, ab.metrics.per_chain(diag), q0, 0.1, draws, T, group)
    b = _run(ab, kind, model, ab.metrics.per_chain(dense), q0, 0.1, draws, T, group)
    for k in a:
        np.testing.assert_array_equal(b[k], a[k], err_msg=k)


# ---------------------------------------------------------------------------------------------------------------------
# 5. NUTS / HMC parity with the oracle run chain by chain
# ---------------------------------------------------------------------------------------------------------------------
def _targets(ab, rng, d):
    if d == "logistic":
        d = 5
        X = np.round(rng.standard_normal((60, d)) * 8) / 8
        y = (rng.random(60) < 0.5).astype(np.float64)
        return ab.models.LogisticRegression(X, y, 2.0), o_models.LogisticRegression(X, y, 2.0), np.zeros(d), d
    mu, cov, prec = _corr_case(rng, d)
    return ab.models.CorrelatedGaussian(mu, prec), o_models.CorrelatedGaussian(mu, prec), mu, d


@pytest.mark.parametrize("group", [8, 32, 256])
@pytest.mark.parametrize("target", [6, 33, "logistic"])
def test_nuts_per_chain_dense_matches_oracle(ab, target, group):
    rng = np.random.default_rng(200 + group + (0 if target == "logistic" else target))
    gm, om, mu, d = _targets(ab, rng, target)
    Cn, T = 70, 3                                        # 70 chains: the last tile of chains is partial
    imms = _spd(rng, Cn, d, 20.0)
    q0 = mu + 0.5 * rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    ref = parity.oracle_nuts(om, q0, 0.15, imms, draws, T, per_chain_imm=True)
    got = _run(ab, "nuts", gm, ab.metrics.per_chain(imms), q0, 0.15, draws, T, group)
    parity.assert_nuts_parity(got, ref, what=f"{target} G={group}")
    np.testing.assert_allclose(got["draws"], ref["draws"], rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("group", [8, 32, 256])
@pytest.mark.parametrize("target", [6, 33, "logistic"])
def test_hmc_per_chain_dense_matches_oracle(ab, target, group):
    rng = np.random.default_rng(300 + group + (0 if target == "logistic" else target))
    gm, om, mu, d = _targets(ab, rng, target)
    Cn, T, L = 70, 3, 4
    imms = _spd(rng, Cn, d, 20.0)
    q0 = mu + 0.5 * rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    ref = parity.oracle_hmc(om, q0, 0.15, imms, draws, T, L, per_chain_imm=True)
    got = _run(ab, "hmc", gm, ab.metrics.per_chain(imms), q0, 0.15, draws, T, group, L=L)
    for k in ("q", "p", "g", "U", "acceptance_probability"):
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-10, atol=1e-12, err_msg=k)
    np.testing.assert_array_equal(got["is_diverging"].astype(bool), ref["is_diverging"].astype(bool))
    np.testing.assert_allclose(got["draws"], ref["draws"], rtol=1e-10, atol=1e-12)


def test_nuts_per_chain_dense_float32_decisions_match(ab):
    rng = np.random.default_rng(9)
    Cn, T, d = 70, 3, 8
    mu, cov, prec = _corr_case(rng, d)
    imms = _spd(rng, Cn, d, 10.0)
    q0 = mu + 0.5 * rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    ref = parity.oracle_nuts(o_models.CorrelatedGaussian(mu, prec), q0, 0.2, imms, draws, T, per_chain_imm=True)
    model = ab.models.CorrelatedGaussian(mu, prec, dtype=torch.float32)
    got = _run(ab, "nuts", model, ab.metrics.per_chain(torch.tensor(imms, dtype=torch.float32)), q0, 0.2, draws, T)
    np.testing.assert_array_equal(got["num_doublings"], ref["num_doublings"])
    np.testing.assert_array_equal(got["n_leapfrog"], ref["n_leapfrog"])
    np.testing.assert_allclose(got["q"], ref["q"], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("L", [1, 2])
def test_hmc_per_chain_dense_single_tick_transitions(ab, L):
    """A transition that lasts one tick starts the next on the following tick: the rider's p0 and v0 of that chain
    (from its own factors) must have landed by then."""
    rng = np.random.default_rng(40 + L)
    Cn, T, d = 70, 5, 12
    gm, om, mu, d = _targets(ab, rng, d)
    imms = _spd(rng, Cn, d, 20.0)
    q0 = mu + rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    ref = parity.oracle_hmc(om, q0, 0.2, imms, draws, T, L, per_chain_imm=True)
    got = _run(ab, "hmc", gm, ab.metrics.per_chain(imms), q0, 0.2, draws, T, L=L)
    for k in ("q", "p", "g", "U", "acceptance_probability"):
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-10, atol=1e-12, err_msg=k)
    np.testing.assert_allclose(got["draws"], ref["draws"], rtol=1e-10, atol=1e-12)


def test_nuts_per_chain_dense_first_step_divergence(ab):
    rng = np.random.default_rng(41)
    Cn, T, d = 70, 4, 10
    gm, om, mu, d = _targets(ab, rng, d)
    imms = _spd(rng, Cn, d, 20.0)
    q0 = mu + rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, T, d)
    eps = np.where(np.arange(Cn) % 3 == 0, 0.2, 50.0)
    ref = parity.oracle_nuts(om, q0, eps, imms, draws, T, div_thr=10.0, per_chain_imm=True)
    assert ref["is_diverging"].astype(bool).sum() >= 30 and (ref["n_leapfrog"] == 1).sum() >= 30
    got = _run(ab, "nuts", gm, ab.metrics.per_chain(imms), q0, eps, draws, T, div_thr=10.0)
    parity.assert_nuts_parity(got, ref)
    np.testing.assert_allclose(got["draws"], ref["draws"], rtol=1e-10, atol=1e-12)


def test_nuts_per_chain_dense_resume_in_chunks_is_bit_exact(ab):
    """A free-running run continued call after call (the chain state machines and the momentum look-ahead stay in
    the workspace) equals the same number of ticks in one call, bit for bit."""
    from aehmc_b200 import _engine
    rng = np.random.default_rng(42)
    Cn, d = 70, 9
    gm, om, mu, d = _targets(ab, rng, d)
    metric = ab.metrics.GaussianMetric(ab.metrics.per_chain(_spd(rng, Cn, d, 20.0)))
    q0 = mu + rng.standard_normal((Cn, d))
    eps = torch.full((Cn,), 0.2, dtype=torch.float64)
    one, ex1 = _engine.run("nuts", gm, metric, ab.RandomStream(seed=3), ab.nuts.new_state(q0, gm), eps,
                           max_ticks=40, group=8)
    key = ("dense-per-chain-resume", Cn)
    srng = ab.RandomStream(seed=3)
    info, ex = _engine.run("nuts", gm, metric, srng, ab.nuts.new_state(q0, gm), eps, max_ticks=10, group=8,
                           workspace_key=key)
    for _ in range(3):
        info, ex = _engine.run("nuts", gm, metric, srng, info.state, ex["step_size"], max_ticks=10, group=8,
                               resume=True, workspace_key=key)
    _engine.release_workspace(key)
    assert torch.equal(info.state.position, one.state.position)
    assert torch.equal(info.state.momentum, one.state.momentum)
    assert torch.equal(info.state.potential_energy_grad, one.state.potential_energy_grad)


# ---------------------------------------------------------------------------------------------------------------------
# 6. window adaptation against the reference's is_mass_matrix_full=True, per chain
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["nuts", "hmc"])
def test_per_chain_dense_warmup_matches_oracle(ab, kind):
    rng = np.random.default_rng(29)
    Cn, W, d, L = 9, 25, 4, 5
    mu, cov, prec = _corr_case(rng, d)
    q0 = mu + rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, W, d)
    om = o_models.CorrelatedGaussian(mu, prec)
    q_ref, eps_ref, imm_ref = [], [], []
    for c in range(Cn):
        if kind == "nuts":
            k = o_kernels.nuts_new_kernel(parity.chain_draws(draws, c), om)
        else:
            hk = o_kernels.hmc_new_kernel(parity.chain_draws(draws, c), om)
            k = lambda s, e, m, hk=hk: hk(s, e, m, L)
        with np.errstate(all="ignore"):
            st, (e, m), _ = o_adapt.run(k, o_kernels.new_state(q0[c].copy(), om), W, is_mass_matrix_full=True)
        q_ref.append(st.position); eps_ref.append(e); imm_ref.append(m)
    model = ab.models.CorrelatedGaussian(mu, prec)
    if kind == "nuts":
        srng = ab.InjectedDraws(**{k: draws[k] for k in ("z", "u_dir", "u_biased", "u_uniform")})
        kernel, state, kw = ab.nuts.new_kernel(srng, model), ab.nuts.new_state(q0, model), {}
    else:
        srng = ab.InjectedDraws(z=draws["z"], u_accept=draws["u_accept"])
        kernel, state, kw = ab.hmc.new_kernel(srng, model), ab.hmc.new_state(q0, model), {"num_integration_steps": L}
    state, (eps, imm), _ = ab.window_adaptation.run(kernel, state, W, is_mass_matrix_full=True, **kw)
    assert imm.shape == (Cn, d, d) and eps.shape == (Cn,)
    np.testing.assert_allclose(_np(imm), np.array(imm_ref), rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(_np(eps), np.array(eps_ref), rtol=1e-6)
    np.testing.assert_allclose(_np(state.position), np.array(q_ref), rtol=1e-5, atol=1e-8)


def test_composed_per_chain_dense_warmup_runs_for_many_chains(ab):
    """A kernel without ``spec`` (the composed path) adapts a dense matrix per chain instead of raising."""
    rng = np.random.default_rng(30)
    Cn, W, d = 4, 25, 3
    mu, cov, prec = _corr_case(rng, d)
    q0 = mu + rng.standard_normal((Cn, d))
    draws = parity.random_draws(rng, Cn, W, d)
    model = ab.models.CorrelatedGaussian(mu, prec)
    srng = ab.InjectedDraws(**{k: draws[k] for k in ("z", "u_dir", "u_biased", "u_uniform")})
    inner = ab.nuts.new_kernel(srng, model)
    kernel = lambda s, e, m: inner(s, e, m)
    state, (eps, imm), _ = ab.window_adaptation.run(kernel, ab.nuts.new_state(q0, model), W, is_mass_matrix_full=True)
    assert imm.shape == (Cn, d, d)
    srng2 = ab.InjectedDraws(**{k: draws[k] for k in ("z", "u_dir", "u_biased", "u_uniform")})
    state2, (eps2, imm2), _ = ab.window_adaptation.run(ab.nuts.new_kernel(srng2, model), ab.nuts.new_state(q0, model),
                                                       W, is_mass_matrix_full=True)
    np.testing.assert_allclose(_np(imm), _np(imm2), rtol=1e-7)
    np.testing.assert_allclose(_np(eps), _np(eps2), rtol=1e-7)


# ---------------------------------------------------------------------------------------------------------------------
# 7. statistics with the native RNG
# ---------------------------------------------------------------------------------------------------------------------
def test_per_chain_dense_warmup_recovers_covariance_and_cuts_leapfrogs(ab):
    """1024 chains, d = 16, covariance with eigenvalues log-spaced over [1e-3, 1] in a random orientation, 300 warm-up
    steps: the last slow window holds n = 100 draws of each chain.  For n independent draws the sample covariance S
    has E ||S - Sigma||_F^2 = (tr(Sigma)^2 + tr(Sigma^2)) / n; the bound on the median relative error allows an
    effective sample size of n / 3 (the draws of one chain are correlated, and the window samples with the previous
    window's metric).  Sampling with the adapted dense matrices then needs at most half the leapfrogs per transition
    of per-chain diagonal adaptation, which cannot undo the rotation."""
    rng = np.random.default_rng(77)
    Cn, d, W = 1024, 16, 300
    cov = _spd(rng, 1, d, 1e3)[0]
    model = ab.models.CorrelatedGaussian(np.zeros(d), np.linalg.inv(cov))
    q0 = rng.standard_normal((Cn, d)) * 0.1
    mean_lf = {}
    for full in (True, False):
        kernel = ab.nuts.new_kernel(ab.RandomStream(seed=5), model)
        state, (eps, imm), _ = ab.window_adaptation.run(kernel, ab.nuts.new_state(q0, model), W,
                                                        is_mass_matrix_full=full)
        if full:
            assert imm.shape == (Cn, d, d)
            err = np.linalg.norm(_np(imm) - cov, axis=(1, 2)) / np.linalg.norm(cov)
            bound = np.sqrt(3.0 * (np.trace(cov) ** 2 + np.trace(cov @ cov)) / 100.0) / np.linalg.norm(cov)
            assert np.median(err) < bound, (np.median(err), bound)
        _, _, stats, _ = ab.sampling.sample(kernel, state, eps, ab.metrics.per_chain(imm), 100)
        mean_lf[full] = float(stats[:, :, 2].mean())
    assert mean_lf[True] <= 0.5 * mean_lf[False], mean_lf


# ---------------------------------------------------------------------------------------------------------------------
# 8. checkpoints and errors
# ---------------------------------------------------------------------------------------------------------------------
def test_checkpoint_restore_per_chain_dense_is_bit_exact(ab):
    rng = np.random.default_rng(12)
    Cn, d = 64, 8
    mu, cov, prec = _corr_case(rng, d)
    model = ab.models.CorrelatedGaussian(mu, prec)
    imm = ab.metrics.per_chain(torch.tensor(_spd(rng, Cn, d, 20.0), device="cuda"))
    q0 = mu + rng.standard_normal((Cn, d))
    whole = ab.sampling.sample(ab.nuts.new_kernel(ab.RandomStream(seed=9), model), ab.nuts.new_state(q0, model), 0.3,
                               imm, 6)
    srng1 = ab.RandomStream(seed=9)
    first = ab.sampling.sample(ab.nuts.new_kernel(srng1, model), ab.nuts.new_state(q0, model), 0.3, imm, 3)
    buf = io.BytesIO()
    torch.save(ab.sampling.checkpoint(first[0].state, srng1, 0.3, ab.metrics.GaussianMetric(imm)), buf)
    buf.seek(0)
    ck = torch.load(buf, weights_only=False)
    assert ck["inverse_mass_matrix_kind"] == "per_chain" and tuple(ck["inverse_mass_matrix"].shape) == (Cn, d, d)
    state, srng2, eps, imm2 = ab.sampling.restore(ck, device="cuda:0")
    assert isinstance(imm2, ab.metrics.per_chain)
    second = ab.sampling.sample(ab.nuts.new_kernel(srng2, model), state, eps, imm2, 3)
    assert torch.equal(torch.cat([first[1], second[1]]), whole[1])
    assert torch.equal(second[0].state.position, whole[0].state.position)


def test_per_chain_dense_errors(ab):
    from aehmc_b200 import _engine, _lib, backend
    rng = np.random.default_rng(13)
    Cn, d = 6, 5
    mu, cov, prec = _corr_case(rng, d)
    model = ab.models.CorrelatedGaussian(mu, prec)
    q0 = mu + rng.standard_normal((Cn, d))
    wrong = ab.metrics.per_chain(_spd(rng, Cn + 1, d))
    with pytest.raises(ValueError, match="chains, dim, dim"):
        _engine.run("nuts", model, wrong, ab.RandomStream(1), ab.nuts.new_state(q0, model), 0.2)
    with pytest.raises(ValueError, match="pooled=True"):
        ab.metrics.gaussian_metric(ab.metrics.per_chain(torch.eye(129, dtype=torch.float64).expand(2, 129, 129)))
    # the C-ABI: d beyond the limit, and the entry points that reject every dense kind
    big = ab.models.IIDGaussian(np.zeros(129), np.ones(129))
    t = torch.zeros(4 * 129 * 129, dtype=torch.float64, device="cuda")
    m = _lib.Metric(_lib.IMM_DENSE_PER_CHAIN, 1, 0.0, t.data_ptr(), t.data_ptr(), t.data_ptr())
    cfg = _lib.Cfg(_lib.F64, 10, 1000.0, 0, 0, 0, 1, 0, 0)
    lib = _lib.load()
    assert lib.b2h_nuts_workspace_bytes(C.byref(big.struct()), C.byref(m), C.byref(cfg), C.c_int64(2)) < 0
    ctx = backend.context(t.device)
    zero = torch.zeros(64, dtype=torch.int64, device="cuda")
    rc = lib.b2h_is_iterative_turning(ctx, C.byref(m), _lib.F64, backend.ptr(t), backend.ptr(t), backend.ptr(zero),
                                      backend.ptr(zero), backend.ptr(t), backend.ptr(t), backend.ptr(zero),
                                      C.c_int64(2), C.c_int64(d), C.c_int32(10))
    assert rc == -3
    small = ab.models.CorrelatedGaussian(mu, prec).struct()
    rng_s = _lib.Rng()
    tree, sub = _lib.Tree(), _lib.Subtree()
    eps = torch.ones(2, dtype=torch.float64, device="cuda")
    assert lib.b2h_nuts_expand(ctx, C.byref(small), C.byref(m), C.byref(rng_s), C.byref(cfg), C.byref(tree),
                               backend.ptr(eps), C.c_int64(2), None, backend.ptr(t), C.c_int64(t.numel() * 8)) == -3
    sub.max_num_steps = 1
    assert lib.b2h_nuts_subtree(ctx, C.byref(small), C.byref(m), C.byref(rng_s), C.byref(cfg), C.byref(sub),
                                backend.ptr(eps), C.c_int64(2), backend.ptr(t), C.c_int64(t.numel() * 8)) == -3
