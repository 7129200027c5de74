"""Potential and gradient of the fp16 x 2 fused logistic gradient, written as .npy files for a byte comparison of two
builds of the library (B2H_LIB selects one).  Shapes: the c5 shape (131072 chains, N = 100000, D = 128: the KB = 2
kernel, a partial last data tile) and a D = 64 shape (the KB = 1 kernel), seeded positions.
    python benchmarks/fused16_grad_dump.py OUTDIR"""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
import aehmc_b200 as ab

out = sys.argv[1]
os.makedirs(out, exist_ok=True)
for name, chains, n, d in (("c5", 131072, 100000, 128), ("d64", 16384, 100000, 64)):
    X, y, _ = bench.make_logistic_problem(n, d)
    model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float32, tensor_core=True)
    assert model.tc_flag == 4.0, model.tc_flag
    q = bench.initial_positions("logistic", chains, d) + 0.01 * np.random.default_rng(9).standard_normal((chains, d))
    U, g = model.potential_and_grad(torch.tensor(q, dtype=torch.float32, device="cuda"))
    torch.cuda.synchronize()
    np.save(os.path.join(out, f"{name}_U.npy"), U.cpu().numpy())
    np.save(os.path.join(out, f"{name}_g.npy"), g.cpu().numpy())
    print(name, "U sum", float(U.double().sum()), "g abs sum", float(g.double().abs().sum()))
