"""The grouped dense contraction of csrc/gemm.cu (b2h_gemm) against an exact reference, on every dispatch path.

The kernel behind the dense mass-matrix apply, the correlated-Gaussian gradient, the momentum contractions of
restarting chains and the pooled second moment chooses among: the FP64 cp.async DMMA kernel at tile width
BN = 96 / 112 / 128 (BN = 112: an odd number of n8 tiles per warp), split-K partial planes, device-side row counts
(the LOOP kernel, whose CTAs walk several row tiles), up to three groups, triangular B, the subtracted vector, the
register-staged DMMA kernel (unaligned rows or pointers) and the FP32 SIMT kernel.

Exactness: integer-valued inputs keep every partial sum exact in any summation order, so the kernel must equal the
float64 product bit for bit.  Random-normal FP64 cases are checked against the standard dot-product bound
|err| <= 1.01 (K + 2) 2^-53 (|A - sub| |B|) with an extended-precision reference (a silent drop to FP32 or TF32
arithmetic misses it by orders of magnitude).

Edges: everything outside the logical A, B and sub is NaN (a read past an edge that reaches the arithmetic makes the
result NaN), and the output buffer holds one plane more than the launch writes, with wider rows, pre-filled with a
sentinel that must survive everywhere outside rows < min(M, count), columns < N and planes < nsplit.

The environment-selected variants (B2H_GEMM_BN, B2H_GEMM_WARPS, B2H_GEMM_BK, B2H_GEMM_ASYNC with B2H_DMMA_K) are read
once per process, so each one re-runs the case list in a child process (this file run as a script).
"""
import ctypes as C
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BM = 128
SMS = 148
DEVICE = "cuda:0"
ENV_KEYS = ("B2H_GEMM_BN", "B2H_GEMM_WARPS", "B2H_GEMM_BK", "B2H_GEMM_ASYNC", "B2H_DMMA_K")
SENTINEL = {"f64": -1.25e300, "f32": -1.25e30}


def pick_bn(M0, N):
    """gemm.cu pick_bn (no rider tile rows): the width whose tile count wastes the least of the last wave."""
    best, best_cost = 128, 1e300
    for bn in (128, 112, 96):
        tiles = ((M0 + BM - 1) // BM) * ((N + bn - 1) // bn)
        cost = ((tiles + SMS - 1) // SMS) * bn
        if cost < best_cost - 1e-9:
            best, best_cost = bn, cost
    return best


def empty_slices(K, nsplit):
    """Split-K slices without a k-range (non-triangular launch): k_chunk = ceil(K / nsplit) rounded up to 16."""
    chunk = (K + nsplit - 1) // nsplit
    chunk = (chunk + 15) // 16 * 16
    return [s for s in range(nsplit) if s * chunk >= K]


def grp(M, count=None, sub=False, tri=0, lda_pad=2, a_off=0):
    return dict(M=M, count=count, sub=sub, tri=tri, lda_pad=lda_pad, a_off=a_off)


def case(name, dtype, N, K, groups, nsplit=1, vals="int", ldb_pad=2, ldo_pad=2, shared_a=False, heuristic=False,
         expect_bn=None):
    return dict(name=name, dtype=dtype, N=N, K=K, groups=groups, nsplit=nsplit, vals=vals, ldb_pad=ldb_pad,
                ldo_pad=ldo_pad, shared_a=shared_a, heuristic=heuristic, expect_bn=expect_bn)


def build_cases():
    cs = []
    Ms, Ns, Ks = (1, 127, 128, 129, 1000), (2, 16, 96, 112, 113, 128, 130, 1000), (2, 30, 32, 34, 1000)
    # edges by default dispatch: every N against every K, M cycling through its edge values, with and without sub
    for dt in ("f64", "f32"):
        for i, N in enumerate(Ns):
            for j, K in enumerate(Ks):
                M = Ms[(i + 2 * j) % len(Ms)]
                for s in (False, True):
                    vals = "large" if dt == "f64" and (i + j) % 2 else "int"
                    cs.append(case(f"edge-{dt}-M{M}-N{N}-K{K}-{'sub' if s else 'nosub'}", dt, N, K, [grp(M, sub=s)],
                                   vals=vals))
        # register-staged fallback: odd N or K, odd lda, A pointer off by one element
        for M, N, K, lp, off in ((129, 17, 34, 2, 0), (200, 34, 17, 1, 0), (129, 999, 999, 2, 0), (300, 130, 32, 1, 0),
                                 (257, 112, 1000, 3, 0), (129, 128, 64, 2, 1), (1000, 113, 30, 2, 1)):
            for s in (False, True):
                cs.append(case(f"fallback-{dt}-M{M}-N{N}-K{K}-lda+{lp}-off{off}-{'sub' if s else 'nosub'}", dt, N, K,
                               [grp(M, sub=s, lda_pad=lp, a_off=off)]))
        # split-K: the planes sum to the product; slices without a k-range write exact zeros
        for ns in (1, 2, 3, 5, 8):
            for K in (34, 100, 1000):
                cs.append(case(f"split-{dt}-K{K}-ns{ns}", dt, 130, K, [grp(129, sub=(ns + K) % 2 == 1)], nsplit=ns))
        # device row counts: LOOP walk (count above M clamps to M)
        for cnt in (0, 1, 127, 128, 129, 4095, 4096, 5000):
            cs.append(case(f"count-{dt}-{cnt}", dt, 128, 128, [grp(4096, count=cnt, sub=cnt % 2 == 1)]))
        for ns in (1, 5):   # 313 row tiles against at most 296 CTAs (60 at nsplit 5): CTAs walk several tiles
            cs.append(case(f"walk-{dt}-40000-ns{ns}", dt, 128, 128, [grp(40000, count=40000, sub=ns == 5)], nsplit=ns))
        cs.append(case(f"groups3-{dt}-300-0-129", dt, 130, 96,
                       [grp(1000, count=300, sub=True), grp(500, count=0), grp(700, count=129)]))
        cs.append(case(f"groups3-{dt}-300-0-129-ns3", dt, 130, 100,
                       [grp(1000, count=300), grp(500, count=0, sub=True), grp(700, count=129)], nsplit=3))
        cs.append(case(f"static+count-{dt}", dt, 112, 200, [grp(200, sub=True), grp(1000, count=300)]))
        cs.append(case(f"count+static-{dt}-ns2", dt, 112, 200, [grp(1000, count=129), grp(300)], nsplit=2))
        # triangular B: tri = 1 upper, tri = 2 lower (non-zero diagonal and triangle)
        for d in (300, 1000):
            for ns in (1, 5):
                for tri in (1, 2):
                    cs.append(case(f"tri{tri}-{dt}-d{d}-ns{ns}", dt, d, d, [grp(129 if d == 1000 else 257, tri=tri,
                                                                                 sub=ns == 5)], nsplit=ns))
            # the momentum contractions of restarting chains: one A, lower (tri 2) and upper (tri 1) factor, one
            # device count, 5 split-K slices
            cs.append(case(f"rider-{dt}-d{d}", dt, d, d, [grp(4096 if d == 1000 else 600, count=385, tri=2),
                                                         grp(4096 if d == 1000 else 600, count=385, tri=1)],
                           nsplit=5, shared_a=True))
        cs.append(case(f"tri-fallback-{dt}", dt, 300, 300, [grp(257, tri=2, lda_pad=1), grp(100, tri=1, lda_pad=1)],
                       nsplit=3))
    # random-normal FP64, one per path (extended-precision reference on a subset of rows)
    cs += [
        case("normal-bn96", "f64", 130, 130, [grp(129, sub=True)], vals="normal"),
        case("normal-fallback", "f64", 130, 131, [grp(129, sub=True, lda_pad=1)], vals="normal"),
        case("normal-split5", "f64", 130, 1000, [grp(129, sub=True)], nsplit=5, vals="normal"),
        case("normal-count", "f64", 128, 500, [grp(4096, count=777, sub=True)], vals="normal"),
        case("normal-walk", "f64", 128, 128, [grp(40000, count=40000)], nsplit=5, vals="normal"),
        case("normal-rider", "f64", 1000, 1000, [grp(4096, count=385, tri=2), grp(4096, count=385, tri=1)], nsplit=5,
             vals="normal", shared_a=True),
        case("normal-f32", "f32", 130, 1000, [grp(129, sub=True)], nsplit=2, vals="normal"),
    ]
    # tile widths reached by the default heuristic (left out of the forced-variant runs)
    cs += [
        case("c2-shape-bn112", "f64", 1000, 1000, [grp(4096)], vals="large", heuristic=True, expect_bn=112),
        case("c2-shape-bn112-sub", "f64", 1000, 1000, [grp(4096, sub=True)], heuristic=True, expect_bn=112),
        case("wide-bn128", "f64", 128, 128, [grp(131072, sub=True)], vals="large", heuristic=True, expect_bn=128),
        case("normal-bn112", "f64", 1000, 1000, [grp(2048, sub=True)], vals="normal", heuristic=True, expect_bn=112),
        case("normal-bn128", "f64", 128, 128, [grp(12800)], vals="normal", heuristic=True, expect_bn=128),
    ]
    names = [c["name"] for c in cs]
    assert len(names) == len(set(names))
    return cs


CASES = build_cases()


def _ints(rng, shape, lim, nonzero=False):
    x = rng.integers(-lim, lim + 1, size=shape).astype(np.float64)
    if nonzero:
        x[x == 0] = 1.0
    return x


def _values(rng, c, shape, role, nonzero=False):
    """role 'a' (A and sub), 'b' (B).  Integer ranges keep K max|a - sub| max|b| below 2^53 (FP64) / 2^24 (FP32)."""
    if c["vals"] == "normal":
        x = rng.standard_normal(shape)
        return x.astype(np.float32).astype(np.float64) if c["dtype"] == "f32" else x
    if c["dtype"] == "f32":
        lim = 16 if role == "a" else 32            # 1000 * 32 * 32 < 2^24
    elif c["vals"] == "large":
        lim = 2 ** 19 if role == "a" else 2 ** 20  # 1000 * 2^20 * 2^20 < 2^53
    else:
        lim = 2 ** 9 if role == "a" else 2 ** 10
    return _ints(rng, shape, lim, nonzero)


def _check_rows(c, Mv):
    """Rows whose values are compared (normal data: an extended-precision reference on a subset)."""
    if c["vals"] != "normal" or Mv <= 96:
        return np.arange(Mv)
    rng = np.random.default_rng(7)
    edge = [r for r in (0, 1, 31, 32, 127, 128, 129, 255, 256) if r < Mv] + list(range(max(Mv - 8, 0), Mv))
    return np.unique(np.concatenate([edge, rng.choice(Mv, 48, replace=False)])).astype(np.int64)


def run_case(c, lib, ctx, check_bn=True):
    """Runs one case through b2h_gemm; returns a list of mismatch descriptions (empty: the case passed)."""
    from aehmc_b200 import _lib
    dt = torch.float64 if c["dtype"] == "f64" else torch.float32
    npdt = np.float64 if c["dtype"] == "f64" else np.float32
    dev = torch.device(DEVICE)
    rng = np.random.default_rng(zlib.crc32(c["name"].encode()))
    N, K, ns = c["N"], c["K"], c["nsplit"]
    ldb, ldo = N + c["ldb_pad"], N + c["ldo_pad"]
    errs = []
    if check_bn and c["expect_bn"] is not None and pick_bn(c["groups"][0]["M"], N) != c["expect_bn"]:
        errs.append(f"{c['name']}: the heuristic now picks BN = {pick_bn(c['groups'][0]['M'], N)}, "
                    f"the case was meant to cover BN = {c['expect_bn']}")
    keep, host = [], []
    structs = (_lib.GemmGroup * 3)()
    split_stride = max((g["M"] + 3) * ldo for g in c["groups"]) + 2
    for gi, g in enumerate(c["groups"]):
        M = g["M"]
        src = host[0] if (c["shared_a"] and gi > 0) else None
        if src is None:
            lda = K + g["lda_pad"]
            a = _values(rng, c, (M, K), "a")
            s = _values(rng, c, (K,), "a") if g["sub"] else None
            abuf = torch.full(((M + 3) * lda + g["a_off"],), float("nan"), dtype=dt)
            abuf[g["a_off"]:].view(M + 3, lda)[:M, :K] = torch.from_numpy(a)
            abuf = abuf.to(dev)
            A = abuf[g["a_off"]:]
            sbuf = None
            if s is not None:
                sbuf = torch.full((K + 4,), float("nan"), dtype=dt)
                sbuf[:K] = torch.from_numpy(s)
                sbuf = sbuf.to(dev)
            cnt = None
            if g["count"] is not None:
                cnt = torch.tensor([g["count"]], dtype=torch.int32, device=dev)
            keep += [abuf, sbuf, cnt]
        else:
            a, s, lda, A, sbuf, cnt = src["a"], src["s"], src["lda"], src["A"], src["sbuf"], src["cnt"]
        b = _values(rng, c, (K, N), "b", nonzero=g["tri"] != 0)
        if g["tri"] == 1:
            b = np.triu(b)          # B[k][n] = 0 for k > n
        elif g["tri"] == 2:
            b = np.tril(b)          # B[k][n] = 0 for k < n
        bbuf = torch.full((K + 3, ldb), float("nan"), dtype=dt)
        bbuf[:K, :N] = torch.from_numpy(b)
        bbuf = bbuf.to(dev)
        obuf = torch.full(((ns + 1) * split_stride,), SENTINEL[c["dtype"]], dtype=dt, device=dev)
        keep += [bbuf, obuf]
        host.append(dict(a=a, s=s, lda=lda, A=A, sbuf=sbuf, cnt=cnt, b=b, obuf=obuf))
        st = structs[gi]
        st.A, st.lda, st.B, st.ldb = A.data_ptr(), lda, bbuf.data_ptr(), ldb
        st.out, st.ldo, st.M = obuf.data_ptr(), ldo, M
        st.m_dev = cnt.data_ptr() if cnt is not None else None
        st.sub = sbuf.data_ptr() if sbuf is not None else None
        st.tri = g["tri"]
    rc = lib.b2h_gemm(ctx, C.c_int(1 if c["dtype"] == "f64" else 0), structs, C.c_int32(len(c["groups"])),
                      C.c_int64(N), C.c_int64(K), C.c_int32(ns), C.c_int64(split_stride))
    torch.cuda.synchronize()
    if rc != 0:
        return errs + [f"{c['name']}: b2h_gemm returned {rc}: {lib.b2h_last_error()}"]
    sent = npdt(SENTINEL[c["dtype"]])
    empties = empty_slices(K, ns) if all(g["tri"] == 0 for g in c["groups"]) else []
    for gi, (g, h) in enumerate(zip(c["groups"], host)):
        tag = f"{c['name']} group {gi}"
        M = g["M"]
        Mv = M if g["count"] is None else max(0, min(M, g["count"]))
        o = h["obuf"].cpu().numpy()
        planes = o[:(ns + 1) * split_stride].reshape(ns + 1, split_stride)
        grid = np.zeros((ns + 1, M + 3, ldo), dtype=bool)
        grid[:ns, :Mv, :N] = True
        inside = np.zeros((ns + 1, split_stride), dtype=bool)
        inside[:, :(M + 3) * ldo] = grid.reshape(ns + 1, -1)
        if not np.all(planes[~inside] == sent):
            bad = np.argwhere((planes != sent) & ~inside)
            errs.append(f"{tag}: {len(bad)} writes outside the result, first (plane, offset) {bad[:4].tolist()}")
        vals = planes[:ns, :(M + 3) * ldo].reshape(ns, M + 3, ldo)[:, :Mv, :N]
        if np.any(vals == sent):
            errs.append(f"{tag}: {int(np.sum(vals == sent))} result elements never written")
            continue
        if np.isnan(vals).any():
            errs.append(f"{tag}: NaN in the result (a read past an edge of A, B or sub)")
            continue
        for s_ in empties:
            if not np.all(vals[s_] == 0.0):
                errs.append(f"{tag}: slice {s_} has no k-range but its plane is not exactly zero")
        if Mv == 0:
            continue
        rows = _check_rows(c, Mv)
        a = h["a"][rows] - (h["s"] if h["s"] is not None else 0.0)
        if c["vals"] == "normal":
            ld = np.longdouble
            al = h["a"][rows].astype(ld) - (h["s"].astype(ld) if h["s"] is not None else ld(0))
            ref = al @ h["b"].astype(ld)
            got = vals[:, rows].astype(ld).sum(axis=0)
            eps = 2.0 ** -53 if c["dtype"] == "f64" else 2.0 ** -24
            bound = 1.01 * (K + 2) * eps * (np.abs(al) @ np.abs(h["b"]).astype(ld))
            err = np.abs(got - ref)
            if not np.all(err <= bound):
                i = np.unravel_index(np.argmax(err - bound), err.shape)
                errs.append(f"{tag}: error {float(err[i]):.3e} above the bound {float(bound[i]):.3e} at row "
                            f"{rows[i[0]]}, column {i[1]}")
        else:
            ref = a @ h["b"]
            got = vals[:, rows].astype(np.float64).sum(axis=0)
            if not np.array_equal(got, ref):
                bad = np.argwhere(got != ref)
                r, col = bad[0]
                errs.append(f"{tag}: {len(bad)} elements differ from the exact product, first at row {rows[r]}, "
                            f"column {col}: {got[r, col]!r} != {ref[r, col]!r}")
    return errs


def _context():
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    lib.b2h_gemm.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int64]
    return lib, backend.context(torch.device("cuda:0"))


@pytest.fixture(scope="module")
def gemm(cuda_device):
    for k in ENV_KEYS:
        if k in os.environ:
            pytest.skip(f"{k} is set: the default-dispatch cases need the default kernel choice")
    return _context()


@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_gemm_default_dispatch(gemm, c):
    errs = run_case(c, *gemm)
    assert not errs, "\n".join(errs)


def test_heuristic_widths_are_the_shipped_ones():
    """The c2 contraction (4096 chains x d = 1000) runs at BN = 112 and the 131072 x 128 apply at BN = 128."""
    assert pick_bn(4096, 1000) == 112
    assert pick_bn(131072, 128) == 128
    assert empty_slices(34, 8) == [3, 4, 5, 6, 7]


VARIANTS = [{"B2H_GEMM_BN": "96"}, {"B2H_GEMM_BN": "112"}, {"B2H_GEMM_BN": "128"}, {"B2H_GEMM_WARPS": "16"},
            {"B2H_GEMM_BK": "16"}, {"B2H_GEMM_ASYNC": "0", "B2H_DMMA_K": "4"},
            {"B2H_GEMM_ASYNC": "0", "B2H_DMMA_K": "8"}, {"B2H_GEMM_ASYNC": "0", "B2H_DMMA_K": "16"}]


VARIANT_IDS = ["-".join(f"{k}={v}" for k, v in x.items()) for x in VARIANTS]


@pytest.fixture(scope="module")
def variant_runs(cuda_device, tmp_path_factory):
    """One child process per variant, all started at once (the library reads these switches once per process);
    every child is waited for, or killed, before the module ends."""
    out = tmp_path_factory.mktemp("gemm_variants")
    flags = ["-s"] if sys.flags.no_user_site else []
    runs = {}
    try:
        for vid, variant in zip(VARIANT_IDS, VARIANTS):
            env = {k: v for k, v in os.environ.items() if k not in ENV_KEYS}
            env.update(variant)
            log = open(out / f"{vid}.log", "w+")
            p = subprocess.Popen([sys.executable, *flags, os.path.abspath(__file__), "--child"], env=env, cwd=ROOT,
                                 stdout=log, stderr=subprocess.STDOUT, text=True)
            runs[vid] = (p, log)
        yield runs
    finally:
        for p, log in runs.values():
            if p.poll() is None:
                p.kill()
            p.wait()
            log.close()


@pytest.mark.parametrize("vid", VARIANT_IDS)
def test_gemm_forced_variant(variant_runs, vid):
    """The case list, less the shapes that exist only to reach a width by the heuristic, under one environment-selected
    kernel variant."""
    p, log = variant_runs[vid]
    try:
        rc = p.wait(timeout=900)
    except subprocess.TimeoutExpired:
        p.kill()
        p.wait()
        rc = "timeout"
    log.seek(0)
    text = log.read()
    assert rc == 0, f"{vid}: exit {rc}\n{text[-8000:]}"
    assert json.loads(text.strip().splitlines()[-1])["cases"] > 100


def test_gemm_rejects_bad_arguments(gemm):
    lib, ctx = gemm
    buf = torch.zeros(64 * 64, dtype=torch.float64, device="cuda")

    def call(ctx_=ctx, dtype=1, n_groups=1, N=8, K=8, nsplit=1, **over):
        g = (_lib_group() * 3)()
        g[0].A, g[0].B, g[0].out = buf.data_ptr(), buf.data_ptr(), buf.data_ptr()
        g[0].lda, g[0].ldb, g[0].ldo, g[0].M = 8, 8, 8, 8
        for k, v in over.items():
            setattr(g[0], k, v)
        return lib.b2h_gemm(ctx_, C.c_int(dtype), g, C.c_int32(n_groups), C.c_int64(N), C.c_int64(K),
                            C.c_int32(nsplit), C.c_int64(0))

    assert call() == 0
    torch.cuda.synchronize()
    bad = [dict(ctx_=None), dict(dtype=7), dict(n_groups=0), dict(n_groups=4), dict(N=0), dict(K=0), dict(nsplit=0),
           dict(lda=7), dict(ldb=7), dict(ldo=7), dict(M=2 ** 31), dict(M=-1), dict(tri=3)]
    for kw in bad:
        assert call(**kw) == -1, kw


def _lib_group():
    from aehmc_b200 import _lib
    return _lib.GemmGroup


def _child():
    """Runs the case list with the kernel choice the environment selects; prints mismatches and a JSON summary."""
    sys.path.insert(0, ROOT)
    torch.cuda.set_device(0)
    lib, ctx = _context()
    cases = [c for c in CASES if not c["heuristic"]]
    errs = []
    for c in cases:
        errs += run_case(c, lib, ctx, check_bn=False)
    for e in errs:
        print(e)
    print(json.dumps({"cases": len(cases), "failures": len(errs)}))
    return 1 if errs else 0


if __name__ == "__main__" and "--child" in sys.argv:
    sys.exit(_child())
