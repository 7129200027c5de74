"""Host-side helpers of bench.py: synthetic problems are deterministic, bf16 rounding matches torch, the reference arm's
sample shrinks with the number of requested steps, and every workload has a description naming its BASELINE config."""
import numpy as np
import pytest

import bench


def test_bf16_round_matches_torch():
    torch = pytest.importorskip("torch")
    x = np.random.default_rng(0).standard_normal(4096).astype(np.float32) * np.float32(3.0)
    ours = bench.bf16_round(x)
    theirs = torch.from_numpy(x).bfloat16().float().numpy()
    assert np.array_equal(ours, theirs)


def test_problems_are_deterministic_and_well_formed():
    cov, prec = bench.make_dense_problem(16)
    cov2, _ = bench.make_dense_problem(16)
    assert np.array_equal(cov, cov2) and np.allclose(cov @ prec, np.eye(16), atol=1e-9)
    X, y, imm = bench.make_logistic_problem(256, 8)
    assert X.shape == (256, 8) and set(np.unique(y)) <= {0.0, 1.0} and np.allclose(imm, 4.0 / 256)
    assert np.array_equal(bench.bf16_round(X.astype(np.float32)).astype(np.float64), X)      # bf16-representable
    a = bench.initial_positions("logistic", 4, 8, chain_offset=0)
    b = bench.initial_positions("logistic", 4, 8, chain_offset=4)
    assert a.shape == (4, 8) and not np.array_equal(a, b)


def test_reference_arm_sample_is_bounded():
    for name in bench.WORKLOADS:
        full = bench.cpu_transitions(name, 1)
        many = bench.cpu_transitions(name, 50)
        assert 3 <= many <= full
        assert name in bench.describe(name)
    assert "configs[1]" in bench.describe("c2") and "configs[2]" in bench.describe("c3") and "configs[4]" in bench.describe("c5")


@pytest.mark.parametrize("name", ["c5", "c2", "c3small"])
def test_dump_outputs_fixed_sample_float_files_within_64_mb(tmp_path, name):
    """--dump-outputs at the workload's own shape: the same seeded chain sample every time, every file float32 / float64
    and equal to what the engine call returned (integers and flags exactly), all files together within 64 MB."""
    torch = pytest.importorskip("torch")
    from types import SimpleNamespace as NS
    kind, Cn, d, _, _ = bench.WORKLOADS[name]
    dt = torch.float64 if kind == "dense" else torch.float32
    esize = 8 if kind == "dense" else 4
    rows = bench.dump_rows(Cn, d, esize)
    assert np.array_equal(rows, bench.dump_rows(Cn, d, esize)) and np.all(np.diff(rows) > 0) and rows[-1] < Cn
    g = torch.Generator().manual_seed(0)
    st = NS(position=torch.randn((Cn, d), generator=g, dtype=dt), momentum=torch.randn((Cn, d), generator=g, dtype=dt),
            potential_energy=torch.randn(Cn, generator=g, dtype=dt),
            potential_energy_grad=torch.randn((Cn, d), generator=g, dtype=dt))
    info = NS(state=st, acceptance_probability=torch.rand(Cn, generator=g, dtype=torch.float64),
              num_doublings=torch.randint(0, 11, (Cn,), generator=g, dtype=torch.int32),
              is_turning=torch.rand(Cn, generator=g) < 0.5, is_diverging=torch.rand(Cn, generator=g) < 0.1)
    extras = {"n_leapfrog": torch.randint(1, 1024, (Cn,), generator=g, dtype=torch.int32),
              "counters": torch.tensor([123456789012, 4096, 32, Cn * 32], dtype=torch.int64)}
    out = bench.last_step_outputs(info, extras, rows, chain_offset=Cn)
    bench.write_outputs(str(tmp_path), out)
    files = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert set(files) == set(out) and sum(a.nbytes for a in files.values()) <= bench.DUMP_BYTES <= 64 * 10 ** 6
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert np.array_equal(files["chains"], Cn + rows)
    assert np.array_equal(files["position"], st.position.numpy()[rows]) and files["position"].itemsize == esize
    assert np.array_equal(files["potential_energy_grad"], st.potential_energy_grad.numpy()[rows])
    assert np.array_equal(files["num_doublings"], info.num_doublings.numpy()) and np.array_equal(files["is_turning"], info.is_turning.numpy())
    assert np.array_equal(files["counters"], [123456789012, 4096, 32, Cn * 32])
    with pytest.raises(ValueError):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_BYTES // 8 + 1)})


def test_elementwise_roofline_arithmetic():
    """The HBM roofline of the tick kernel: algorithmic bytes 11 d s C over the measured launch time; the traffic figures
    come from the committed profile table (profiles/r02_traffic.json), never from a constant in bench.py."""
    tick = {"avg_launch_us": 300.0, "launches": 62}
    row = bench.elementwise_roofline(tick, "c5", 131072, 128, 4, 32, rest_ms=10.0, hbm_peak=6547.8)
    alg = 11.0 * 128 * 4 * 131072
    assert row["algorithmic_bytes_per_launch"] == alg
    assert abs(row["achieved"] - alg / 300e-6 / 1e9) < 1e-6 and abs(row["frac"] - row["achieved"] / 6547.8) < 1e-12
    assert row["traffic"] is not None and "r02_traffic.json" in row["traffic_from"]
    assert abs(row["traffic_frac"] - row["traffic"] / 300e-6 / 1e9 / 6547.8) < 1e-12
    # without a measured tick kernel (register-front kernels): derived from the step time, and said so
    row2 = bench.elementwise_roofline(None, "c5", 131072, 128, 4, 32, rest_ms=16.0, hbm_peak=6547.8)
    assert row2["how"].startswith("derived") and abs(row2["avg_launch_us"] - 500.0) < 1e-9
