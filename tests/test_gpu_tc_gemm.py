"""The tcgen05 kernels of csrc/tc_gemm.cu against exact or high-precision references, on every dispatch path.

Four kernels and the host code that picks among them:
  * b2h_tc_gemm_bf16: the stand-alone contraction, A-resident kernel (short K, many tiles) or the persistent kernel
    (double-buffered TMEM accumulator, split-K planes);
  * b2h_tc_logistic_residual: the mode-1 epilogue (r = sigmoid(s) - y as three bf16 pieces plus the potential's partial
    sums), first product of the two-kernel logistic gradient;
  * b2h_tc_gemm_blocked_bf16: the second product of the two-kernel gradient (A tile-blocked);
  * the fused bf16 x 3 and fp16 x 2 gradient kernels and the finish kernel, through b2h_potential_and_grad.

Exactness: integer-valued bf16 operands with |a|, |b| <= 16 keep every fp32 partial sum below 2^24, so each split-K
plane must equal the float64 product over its own k-block range bit for bit.  The same holds for the residual pieces
(an exact split of a float32) and for the gradient at q = 0 with integer X.

Edges: everything the kernels must not read is NaN (bf16 NaN in pitch padding, in the rows between M and piece_rows,
after the last row; 0xFF bytes in the workspace, which are NaN as bf16, fp32 and fp64), and outputs are pre-filled
with a sentinel or NaN that must survive wherever nothing is to be written.

The host dispatch formulas are restated in tc_dispatch.py (tc_plan, logreg_tc_plan, fused_plan); a CPU test asserts that the case
list reaches every path.
"""
import ctypes as C
import math
import os
import zlib

import numpy as np
import pytest

from tc_dispatch import (BK, BM, BN, FN, RES_A_BLOCKS, SMS, cdiv, fused_plan, logistic_path, logreg_tc_plan,
                         tc_plan)

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = -1.25e30


# ---------------------------------------------------------------------------------------------------------------
# case lists
# ---------------------------------------------------------------------------------------------------------------
def gcase(name, M, N, K, pieces=1, nsplit=1, rows_pad=0, lda_pad=0, ldb_pad=0):
    return dict(name=name, M=M, N=N, K=K, pieces=pieces, nsplit=nsplit, rows_pad=rows_pad, lda_pad=lda_pad,
                ldb_pad=ldb_pad)


def build_gemm_cases():
    cs = []
    Ms, Ns, Ks = (1, 127, 128, 129, 300), (8, 120, 128, 136, 1000), (8, 16, 56, 64, 72, 136, 1000)
    for i, N in enumerate(Ns):
        for j, K in enumerate(Ks):
            M = Ms[(i + 2 * j) % len(Ms)]
            pieces = 1 + (i + j) % 3
            ns = 1 + (3 * i + j) % 8
            cs.append(gcase(f"edge-M{M}-N{N}-K{K}-p{pieces}-ns{ns}", M, N, K, pieces, ns, rows_pad=8 * ((i + j) % 3),
                            lda_pad=8 * (j % 2), ldb_pad=8 * ((i + 1) % 2)))
    for ns in range(1, 9):
        cs.append(gcase(f"split-K1000-ns{ns}", 129, 136, 1000, 2, ns, rows_pad=8, lda_pad=8, ldb_pad=16))
    cs += [
        gcase("split-kb5-ns4", 300, 200, 300, 3, 4, rows_pad=16),              # 5 k-blocks, 4 asked: 3 planes
        gcase("split-kb3-ns8", 127, 256, 136, 1, 8, lda_pad=8),                  # more slices than k-blocks
        gcase("persistent-3-tiles-per-cta", 2048, 3840, 192, 1, 1, ldb_pad=8),   # 480 tiles on 148 CTAs
        gcase("persistent-4-tiles-per-cta-split", 1024, 2560, 256, 2, 3, rows_pad=8),
        gcase("resident-6-blocks-cross", 300, 12900, 128, 3, 1, rows_pad=8, lda_pad=8, ldb_pad=8),
        gcase("resident-k56-cross", 129, 40000, 56, 1, 1, rows_pad=8, ldb_pad=8),
        gcase("resident-4-blocks", 256, 20000, 128, 2, 1, lda_pad=8),
    ]
    names = [c["name"] for c in cs]
    assert len(names) == len(set(names))
    return cs


def rcase(name, M, N, K, rows_pad=8, s0=False):
    return dict(name=name, M=M, N=N, K=K, rows_pad=rows_pad, s0=s0)


RES_CASES = [rcase("residual-resident-cross", 300, 12900, 128), rcase("residual-persistent-dim136", 200, 1000, 136),
             rcase("residual-persistent-dim64", 129, 1000, 64), rcase("residual-resident-dim8", 1, 38000, 8, rows_pad=0),
             rcase("residual-exact-s0", 129, 1000, 64, s0=True), rcase("residual-exact-s0-resident", 300, 12900, 128, s0=True)]

BLOCKED_CASES = [dict(name="blocked-split5", M=300, N=128, K=1000, nsplit=5),
                 dict(name="blocked-dim136-tail", M=129, N=136, K=900, nsplit=3),
                 dict(name="blocked-chunk-tail", M=300, N=64, K=6480, nsplit=1),
                 dict(name="blocked-kb5-ns4", M=1, N=8, K=300, nsplit=4)]


def fcase(name, mode, dim, N, C_, dtype="f32", vals="normal", misaligned=False):
    return dict(name=name, mode=mode, dim=dim, N=N, C=C_, dtype=dtype, vals=vals, misaligned=misaligned)


def build_fused_cases():
    cs = []
    Ns, Cs = (8, 56, 64, 72, 1000), (1, 127, 129, 4096)
    for mi, mode in enumerate(("fp16x2", "bf16x3", "two_kernel")):
        dims = (8, 16, 56, 64, 72, 120, 128) + ((136, 256) if mode == "two_kernel" else ())
        for i, dim in enumerate(dims):
            N, C_ = Ns[(i + mi) % len(Ns)], Cs[(i + 2 * mi) % len(Cs)]
            dt = "f64" if (i + mi) % 3 == 0 else "f32"
            cs.append(fcase(f"{mode}-d{dim}-N{N}-C{C_}-{dt}", mode, dim, N, C_, dt))
        cs += [
            fcase(f"{mode}-per1-d72", mode, 72, 1000, 129),
            fcase(f"{mode}-planes-d128", mode, 128, 20000, 127, "f64"),
            fcase(f"{mode}-segments-d64", mode, 64, 256, 20000),
            fcase(f"{mode}-C1-d128", mode, 128, 10000, 1),
            fcase(f"{mode}-exact-q0", mode, 64, 1000, 129, "f32", vals="int_q0"),
            fcase(f"{mode}-exact-q0-f64", mode, 128, 72, 4096, "f64", vals="int_q0"),
            fcase(f"{mode}-wrong-labels-d64", mode, 64, 1000, 129, vals="wrong_labels"),
            fcase(f"{mode}-exact-pieces-d128", mode, 128, 40, 129, vals="pieces"),
            fcase(f"{mode}-exact-pieces-d64-f64", mode, 64, 16, 300, "f64", vals="pieces"),
        ]
    cs += [fcase("two_kernel-chunks-d64", "two_kernel", 64, 50000, 4096),
           fcase("two_kernel-d256-C1000", "two_kernel", 256, 1000, 1000, "f64"),
           fcase("fp16x2-misaligned-f32", "fp16x2", 128, 1000, 129, misaligned=True),
           fcase("bf16x3-misaligned-f32", "bf16x3", 64, 1000, 129, misaligned=True)]
    names = [c["name"] for c in cs]
    assert len(names) == len(set(names))
    return cs


GEMM_CASES = build_gemm_cases()
FUSED_CASES = build_fused_cases()


def test_dispatch_coverage():
    """Every path of the host dispatch is reached by at least one case (no GPU needed)."""
    seen = set()
    for c in GEMM_CASES:
        p = tc_plan(c["M"], c["N"], c["K"], c["pieces"], c["nsplit"])
        seen.add(p["kernel"])
        if p["kernel"] == "resident":
            if c["pieces"] * p["kb_total"] == RES_A_BLOCKS:
                seen.add("resident-6-blocks")
            if p["crosses_row_tile"]:
                seen.add("resident-crosses-row-tile")
        else:
            if p["max_tiles_per_cta"] >= 3:
                seen.add("persistent->=3-tiles-per-cta")
            if p["planes"] > 1:
                seen.add("split")
            if c["nsplit"] > p["kb_total"]:
                seen.add("nsplit-above-k-blocks")
            if 1 < p["planes"] < min(c["nsplit"], p["kb_total"]):
                seen.add("nsplit-reduced-by-rounding")
        if c["K"] < BK:
            seen.add("K<64")
        if c["rows_pad"] and c["lda_pad"] and c["ldb_pad"]:
            seen.add("padded-pitches-and-pieces")
    assert {c["nsplit"] for c in GEMM_CASES} == set(range(1, 9))
    assert tc_plan(2048, 3840, 192, 1, 1)["max_tiles_per_cta"] >= 3
    assert tc_plan(300, 200, 300, 3, 4)["planes"] == 3
    for c in RES_CASES:
        seen.add("residual-" + tc_plan(c["M"], c["N"], c["K"], 3, 1)["kernel"])
        if c["N"] % BN:
            seen.add("residual-column-padding")
    for c in BLOCKED_CASES:
        p = tc_plan(c["M"], c["N"], c["K"], 3, c["nsplit"], a_blocked=True)
        assert p["kernel"] == "persistent"
        if p["planes"] > 1:
            seen.add("blocked-split")
        if c["K"] % 128:
            seen.add("blocked-k-tail")
    for c in FUSED_CASES:
        path = logistic_path(c["mode"], c["dim"])
        seen.add(path)
        if path == "two_kernel":
            lp = logreg_tc_plan(c["C"], c["N"], c["dim"])
            if len(lp["chunks"]) >= 2 and lp["chunks"][-1] < lp["n_chunk"]:
                seen.add("two_kernel-chunks-with-tail")
            for nv in lp["chunks"]:
                seen.add("two_kernel-residual-" + tc_plan(c["C"], nv, c["dim"], 3, 1)["kernel"])
            if c["dim"] > 128:
                seen.add("two_kernel-dim>128")
            continue
        fp = fused_plan(c["C"], c["N"])
        kb = cdiv(c["dim"], BK)
        seen.add(f"{path}-KB{kb}")
        if c["C"] == 1:
            seen.add(f"{path}-C1")
        if fp["per_cta"] == 1:
            seen.add(f"{path}-per_cta-1")
        if 1 < fp["per_cta"] < fp["tiles_n"]:
            seen.add(f"{path}-several-planes")
        if fp["per_cta"] > fp["tiles_n"]:
            seen.add(f"{path}-several-segments")
            if fp["boundary_on_chain_tile"]:
                seen.add(f"{path}-boundary-on-chain-tile")
        if c["vals"] == "int_q0":
            seen.add(f"{path}-exact-{c['dtype']}")
        if c["misaligned"]:
            seen.add(f"{path}-misaligned")
    need = {"resident", "persistent", "resident-6-blocks", "resident-crosses-row-tile", "persistent->=3-tiles-per-cta",
            "split", "nsplit-above-k-blocks", "nsplit-reduced-by-rounding", "K<64", "padded-pitches-and-pieces",
            "residual-resident", "residual-persistent", "residual-column-padding", "blocked-split", "blocked-k-tail",
            "two_kernel", "two_kernel-chunks-with-tail", "two_kernel-residual-resident",
            "two_kernel-residual-persistent", "two_kernel-dim>128"}
    for path in ("fused16", "fused"):
        need |= {f"{path}-KB1", f"{path}-KB2", f"{path}-C1", f"{path}-per_cta-1", f"{path}-several-planes",
                 f"{path}-several-segments", f"{path}-boundary-on-chain-tile", f"{path}-exact-f32",
                 f"{path}-exact-f64", f"{path}-misaligned"}
    assert not need - seen, sorted(need - seen)
    # the c5 shape: 131072 chains x N = 100000, about 7 chain-tile segments per CTA, two planes per chain tile
    fp = fused_plan(131072, 100000)
    assert fp["per_cta"] > fp["tiles_n"] and 6 <= fp["per_cta"] / fp["tiles_n"] <= 8 and fp["planes"] == 2


# ---------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------
BF16_NAN = 0x7FC0


def _bf16_bits(x):
    """float64 array of bf16-representable values -> int16 bit patterns (torch, CPU)."""
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).bfloat16().view(torch.int16)


def _bits_to_f64(bits):
    return bits.view(torch.bfloat16).double().numpy()


@pytest.fixture(scope="module")
def tc(cuda_device):
    from aehmc_b200 import _lib, backend
    assert torch.cuda.get_device_properties(0).multi_processor_count == SMS, "the case list is laid out for 148 SMs"
    lib = _lib.load()
    i64, i32, vp = C.c_int64, C.c_int32, C.c_void_p
    lib.b2h_tc_gemm_bf16.argtypes = [vp, vp, i64, vp, i64, vp, i64, i64, i64, i32, i64, i64, i32, i64]
    lib.b2h_tc_logistic_residual.argtypes = [vp, vp, i64, vp, i64, i64, i64, i64, i32, i64, vp, vp, i64, vp, vp]
    lib.b2h_tc_gemm_blocked_bf16.argtypes = [vp, vp, i64, vp, i64, vp, i64, i64, i64, i32, i64, i32, i64]
    return lib, backend.context(torch.device("cuda:0"))


def _ints(rng, shape, lim=16):
    return rng.integers(-lim, lim + 1, size=shape).astype(np.float64)


def _nan_bf16(rows, cols):
    return torch.full((rows, cols), BF16_NAN, dtype=torch.int16)


def _planes_check(tag, o, planes, M, N, ldo, split_stride, ref_planes):
    """o: the whole output buffer (planes + 1 planes of split_stride floats).  Returns mismatch strings."""
    errs = []
    buf = o.reshape(planes + 1, split_stride)
    inside = np.zeros_like(buf, dtype=bool)
    grid = np.zeros((planes + 1, M, ldo), dtype=bool)
    grid[:planes, :, :N] = True
    inside[:, :M * ldo] = grid.reshape(planes + 1, -1)
    if not np.all(buf[~inside] == np.float32(SENTINEL)):
        bad = np.argwhere((buf != np.float32(SENTINEL)) & ~inside)
        errs.append(f"{tag}: {len(bad)} writes outside the result, first (plane, offset) {bad[:4].tolist()}")
    vals = buf[:planes, :M * ldo].reshape(planes, M, ldo)[:, :, :N].astype(np.float64)
    for z in range(planes):
        if not np.array_equal(vals[z], ref_planes[z]):
            bad = np.argwhere(vals[z] != ref_planes[z])
            r, c = bad[0]
            errs.append(f"{tag}: plane {z}: {len(bad)} elements differ from the exact product, first at ({r}, {c}): "
                        f"{vals[z][r, c]!r} != {ref_planes[z][r, c]!r}")
    return errs


def _out_buffer(planes, M, N):
    ldo = (N + 3) // 4 * 4 + 4
    split_stride = (M + 2) * ldo + 4
    return ldo, split_stride, torch.full(((planes + 1) * split_stride,), SENTINEL, dtype=torch.float32, device="cuda")


def run_gemm_case(c, lib, ctx):
    M, N, K, P, ns = c["M"], c["N"], c["K"], c["pieces"], c["nsplit"]
    plan = tc_plan(M, N, K, P, ns)
    rng = np.random.default_rng(zlib.crc32(c["name"].encode()))
    piece_rows = M + c["rows_pad"]
    lda, ldb = (K + 7) // 8 * 8 + c["lda_pad"], (K + 7) // 8 * 8 + c["ldb_pad"]
    a = _ints(rng, (P, M, K))
    b = _ints(rng, (N, K))
    A = _nan_bf16(P * piece_rows + 3, lda)           # NaN: pitch padding, rows M..piece_rows, rows after the last
    for p in range(P):
        A[p * piece_rows:p * piece_rows + M, :K] = _bf16_bits(a[p])
    B = _nan_bf16(N + 3, ldb)
    B[:N, :K] = _bf16_bits(b)
    A, B = A.cuda(), B.cuda()
    ldo, split_stride, out = _out_buffer(plan["planes"], M, N)
    rc = lib.b2h_tc_gemm_bf16(ctx, A.data_ptr(), lda, B.data_ptr(), ldb, out.data_ptr(), M, N, K, P, piece_rows, ldo,
                              ns, split_stride)
    torch.cuda.synchronize()
    if rc != 0:
        return [f"{c['name']}: b2h_tc_gemm_bf16 returned {rc}: {lib.b2h_last_error()}"]
    asum = a.sum(axis=0)
    ref = []
    for z in range(plan["planes"]):
        k0, k1 = z * plan["kb_per"] * BK, min(K, (z + 1) * plan["kb_per"] * BK)
        ref.append(asum[:, k0:k1] @ b[:, k0:k1].T)
    return _planes_check(c["name"], out.cpu().numpy(), plan["planes"], M, N, ldo, split_stride, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("c", GEMM_CASES, ids=[c["name"] for c in GEMM_CASES])
def test_tc_gemm_exact(tc, c):
    errs = run_gemm_case(c, *tc)
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
def test_tc_entry_points_reject_bad_arguments(tc):
    """Bad sizes, pitches and split strides return B2H_ERR_ARG and launch nothing (the output keeps its sentinel)."""
    lib, ctx = tc
    A = torch.zeros((4 * 256, 256), dtype=torch.int16, device="cuda")
    out = torch.full((8 * 256 * 256,), SENTINEL, dtype=torch.float32, device="cuda")
    base = dict(lda=256, ldb=256, M=128, N=128, K=64, pieces=1, piece_rows=128, ldo=128, nsplit=1, split_stride=128 * 128)

    def gemm(**over):
        a = dict(base, **over)
        return lib.b2h_tc_gemm_bf16(ctx, A.data_ptr(), a["lda"], A.data_ptr(), a["ldb"], out.data_ptr(), a["M"], a["N"],
                                    a["K"], a["pieces"], a["piece_rows"], a["ldo"], a["nsplit"], a["split_stride"])

    bad = [dict(M=0), dict(N=0), dict(K=0), dict(pieces=0), dict(M=-1), dict(M=2 ** 31), dict(piece_rows=127),
           dict(lda=56), dict(ldb=56), dict(ldo=124), dict(K=128, nsplit=2, split_stride=128 * 128 + 2),
           dict(K=128, nsplit=2, split_stride=128 * 127 + 124), dict(K=128, nsplit=2, split_stride=-4),
           dict(pieces=3, piece_rows=2 ** 30)]                     # the last piece's rows lie past 2^31
    for kw in bad:
        assert gemm(**kw) == -1, kw
    torch.cuda.synchronize()
    assert bool((out == SENTINEL).all()), "a rejected call wrote to the output"
    assert gemm(K=128, nsplit=2, split_stride=128 * 128 + 4) == 0
    torch.cuda.synchronize()

    R = torch.zeros((3 * 4 * 128 * 128 + 512,), dtype=torch.int16, device="cuda")
    r_al = (-R.data_ptr()) % 1024 // 2
    Rp = R.data_ptr() + 2 * r_al
    y = torch.zeros(256, dtype=torch.float32, device="cuda")
    up = torch.zeros(4 * SMS * 128, dtype=torch.float64, device="cuda")
    per = C.c_int32(-7)
    rbase = dict(lda=64, ldb=64, M=128, N=256, K=64, pieces=3, piece_rows=128, stride=2 * 128 * 128, y=y.data_ptr())

    def resid(**over):
        a = dict(rbase, **over)
        return lib.b2h_tc_logistic_residual(ctx, A.data_ptr(), a["lda"], A.data_ptr(), a["ldb"], a["M"], a["N"], a["K"],
                                            a["pieces"], a["piece_rows"], a["y"], Rp, a["stride"], up.data_ptr(),
                                            C.byref(per))

    for kw in (dict(M=0), dict(N=0), dict(K=0), dict(pieces=0), dict(piece_rows=127), dict(lda=56), dict(ldb=56),
               dict(stride=2 * 128 * 128 - 8), dict(stride=2 * 128 * 128 + 4), dict(y=y.data_ptr() + 4),
               dict(piece_rows=2 ** 30)):
        assert resid(**kw) == -1, kw
    assert per.value == -7
    assert resid() == 0 and per.value == 0
    torch.cuda.synchronize()

    def blocked(**over):
        a = dict(stride=2 * 128 * 128, ldb=256, M=128, N=64, K=256, pieces=3, ldo=64, nsplit=1, split_stride=0)
        a.update(over)
        return lib.b2h_tc_gemm_blocked_bf16(ctx, Rp, a["stride"], A.data_ptr(), a["ldb"], out.data_ptr(), a["M"], a["N"],
                                            a["K"], a["pieces"], a["ldo"], a["nsplit"], a["split_stride"])

    out.fill_(SENTINEL)
    for kw in (dict(M=0), dict(N=0), dict(K=0), dict(pieces=0), dict(stride=128 * 128), dict(stride=2 * 128 * 128 + 8),
               dict(ldb=248), dict(ldo=60), dict(nsplit=2, split_stride=128 * 64 + 2),
               dict(nsplit=2, split_stride=127 * 64 + 60), dict(stride=128 * 2 ** 30)):
        assert blocked(**kw) == -1, kw
    torch.cuda.synchronize()
    assert bool((out == SENTINEL).all()), "a rejected call wrote to the output"


# ---------------------------------------------------------------------------------------------------------------
# mode-1 epilogue: residual pieces and the potential's partial sums
# ---------------------------------------------------------------------------------------------------------------
def _blocked_view(Rbits, piece, stride, tiles_m, tiles_n):
    """[tiles_m * 128, tiles_n * 128] logical view of one piece of a tile-blocked buffer (int16 bits, CPU)."""
    t = Rbits[piece * stride:piece * stride + tiles_n * tiles_m * BM * BN].reshape(tiles_n, tiles_m, BM, BN)
    return t.permute(1, 2, 0, 3).reshape(tiles_m * BM, tiles_n * BN)


def run_residual_case(c, lib, ctx):
    """S = sum_p A_p X^T with A_p = integers x 2^-6 / 2^-7 and X in {-1, 0, 1}: exact in fp32, |S| < 7.  Checks:
      * the pieces are an exact split: r = p0 + p1 + p2 is a float32, p0 = bf16(r), p1 = bf16(r - p0);
      * |r - (sigmoid(S) - y)| <= 2^-21: the exp2 / reciprocal approximations behind __expf and __fdividef are
        within 2^-22 relative for these arguments, plus four fp32 roundings of values below 1 (the largest error
        measured on a B200 is 1.1e-7, a fifth of the bound; a third piece left out costs up to 2^-17 |r|);
      * s0 cases: A = 0, so S = 0 and sigmoid(0) = 1/2 exactly, and y = 1/2 - t with t a float32 of 24 significant
        bits in [1/4, 1/2): the pieces must add up to t exactly, so any piece lost or cut short shows;
      * columns >= N of rows < M are exactly 0, rows >= M are not written (R is NaN-filled), nothing past the pieces;
      * upart, reduced as upart_reduce_kernel does, is within N 2^-18 (each term: the approximations and three fp32
        roundings of values below 8) + 2^-24 L sum |term| (fp32 partial sums of at most L terms) of
        sum softplus(s) - y s."""
    M, N, K = c["M"], c["N"], c["K"]
    plan = tc_plan(M, N, K, 3, 1)
    tm, tn = plan["tiles_m"], plan["tiles_n"]
    rng = np.random.default_rng(zlib.crc32(c["name"].encode()))
    piece_rows = M + c["rows_pad"]
    a = np.stack([_ints(rng, (M, K), 2) / 64, _ints(rng, (M, K), 1) / 128, _ints(rng, (M, K), 1) / 128])
    x = _ints(rng, (N, K), 1)
    y = (rng.random(N) < 0.5).astype(np.float64)
    if c["s0"]:
        a[:] = 0.0
        t = rng.integers(2 ** 23, 2 ** 24, N) * 2.0 ** -25
        y = 0.5 - t
    A = _nan_bf16(3 * piece_rows + 2, K)
    for p in range(3):
        A[p * piece_rows:p * piece_rows + M] = _bf16_bits(a[p])
    B = _nan_bf16(N + 2, K)
    B[:N] = _bf16_bits(x)
    stride = tn * tm * BM * BN + 512                          # a NaN gap after every piece
    Rbuf = torch.full((3 * stride + 1024,), BF16_NAN, dtype=torch.int16, device="cuda")
    off = (-Rbuf.data_ptr()) % 1024 // 2
    yb = torch.tensor(y, dtype=torch.float32, device="cuda")
    n_up = 4 * max(tn, SMS) * M
    up = torch.full((n_up + 64,), float("nan"), dtype=torch.float64, device="cuda")
    A, B = A.cuda(), B.cuda()
    per = C.c_int32(-1)
    rc = lib.b2h_tc_logistic_residual(ctx, A.data_ptr(), K, B.data_ptr(), K, M, N, K, 3, piece_rows, yb.data_ptr(),
                                      Rbuf.data_ptr() + 2 * off, stride, up.data_ptr(), C.byref(per))
    torch.cuda.synchronize()
    tag = c["name"]
    if rc != 0:
        return [f"{tag}: b2h_tc_logistic_residual returned {rc}: {lib.b2h_last_error()}"]
    errs = []
    if per.value != plan["per"]:
        errs.append(f"{tag}: tiles_per_cta {per.value}, the dispatch formula says {plan['per']}")
    R = Rbuf.cpu()[off:off + 3 * stride]
    if not bool((R.reshape(3, stride)[:, stride - 512:] == BF16_NAN).all()):
        errs.append(f"{tag}: writes past the tiles of a piece")
    views = [_blocked_view(R, p, stride, tm, tn) for p in range(3)]
    if not all(bool((v[M:] == BF16_NAN).all()) for v in views):
        errs.append(f"{tag}: rows >= M were written")
    pad = [_bits_to_f64(v[:M, N:].contiguous()) for v in views]
    if not all(np.all(pp == 0.0) for pp in pad):
        errs.append(f"{tag}: columns >= N of valid rows are not 0")
    p0, p1, p2 = (_bits_to_f64(v[:M, :N].contiguous()) for v in views)
    r = p0 + p1 + p2
    if np.isnan(r).any():
        return errs + [f"{tag}: residual pieces not written"]
    rf = r.astype(np.float32)
    if not np.array_equal(rf.astype(np.float64), r):
        errs.append(f"{tag}: p0 + p1 + p2 is not a float32")
    t0 = torch.from_numpy(rf).bfloat16().double().numpy()
    t1 = torch.from_numpy((rf - t0.astype(np.float32))).bfloat16().double().numpy()
    if not (np.array_equal(t0, p0) and np.array_equal(t1, p1)):
        errs.append(f"{tag}: the pieces are not the rounded split bf16(r), bf16(r - p0), rest")
    S = a.sum(axis=0) @ x.T
    ref = 1.0 / (1.0 + np.exp(-S)) - y
    err = np.abs(r - ref).max()
    RATIOS[tag + " residual"] = err / 2.0 ** -21
    if err > 2.0 ** -21:
        errs.append(f"{tag}: residual error {err:.3e} above 2^-21")
    if c["s0"] and not np.array_equal(r, np.broadcast_to(0.5 - y, r.shape)):
        errs.append(f"{tag}: S = 0: {int(np.sum(r != 0.5 - y))} residuals differ from 1/2 - y")
    # potential partials, reduced like upart_reduce_kernel
    u = up.cpu().numpy()
    term = np.logaddexp(0.0, S) - y * S
    got = np.zeros(M)
    for row in range(M):
        if plan["per"] > 0:
            mt = row // BM
            t0_, t1_ = (mt * tn) // plan["per"] * 4, (((mt + 1) * tn - 1) // plan["per"] + 1) * 4
        else:
            t0_, t1_ = 0, 4 * tn
        got[row] = u[np.arange(t0_, t1_) * M + row].sum()
    L = 32 * max(plan["per"], 1)
    bound = N * 2.0 ** -18 + 2.0 ** -24 * L * np.abs(term).sum(axis=1)
    uerr = np.abs(got - term.sum(axis=1))
    RATIOS[tag + " upart"] = float(np.nanmax(uerr / bound))
    print(f"{tag}: residual error / bound {RATIOS[tag + ' residual']:.4f}, potential partials {RATIOS[tag + ' upart']:.4f}")
    if not np.all(uerr <= bound):
        i = int(np.nanargmax(uerr / bound))
        errs.append(f"{tag}: potential partial sums of row {i}: error {uerr[i]:.3e}, bound {bound[i]:.3e}")
    return errs


RATIOS = {}


@pytest.mark.gpu
@pytest.mark.parametrize("c", RES_CASES, ids=[c["name"] for c in RES_CASES])
def test_tc_logistic_residual(tc, c):
    errs = run_residual_case(c, *tc)
    assert not errs, "\n".join(errs)


def run_blocked_case(c, lib, ctx):
    """out = sum_p R_p . B^T with integer R in the tile-blocked layout: bit for bit per split plane.  Rows >= M of the
    blocked tiles and the gap after each piece are NaN; columns >= K of the last k tile hold integers that must meet
    the zero fill of B's tensor map."""
    M, N, K, ns = c["M"], c["N"], c["K"], c["nsplit"]
    plan = tc_plan(M, N, K, 3, ns, a_blocked=True)
    rng = np.random.default_rng(zlib.crc32(c["name"].encode()))
    tm, tk = cdiv(M, BM), cdiv(K, 128)
    stride = tk * tm * BM * BN + 2 * BN * 8
    r = _ints(rng, (3, tm * BM, tk * 128))
    r[:, M:, :] = np.nan
    R = torch.full((3 * stride + 1024,), BF16_NAN, dtype=torch.int16)
    for p in range(3):
        blk = _bf16_bits(r[p]).reshape(tm, BM, tk, 128).permute(2, 0, 1, 3).reshape(-1)
        R[p * stride:p * stride + blk.numel()] = blk
    ldb = (K + 7) // 8 * 8 + 8
    b = _ints(rng, (N, K))
    B = _nan_bf16(N + 2, ldb)
    B[:N, :K] = _bf16_bits(b)
    R, B = R.cuda(), B.cuda()
    ldo, split_stride, out = _out_buffer(plan["planes"], M, N)
    rc = lib.b2h_tc_gemm_blocked_bf16(ctx, R.data_ptr(), stride, B.data_ptr(), ldb, out.data_ptr(), M, N, K, 3, ldo, ns,
                                      split_stride)
    torch.cuda.synchronize()
    if rc != 0:
        return [f"{c['name']}: b2h_tc_gemm_blocked_bf16 returned {rc}: {lib.b2h_last_error()}"]
    rs = r[:, :M, :K].sum(axis=0)
    ref = []
    for z in range(plan["planes"]):
        k0, k1 = z * plan["kb_per"] * BK, min(K, (z + 1) * plan["kb_per"] * BK)
        ref.append(rs[:, k0:k1] @ b[:, k0:k1].T)
    return _planes_check(c["name"], out.cpu().numpy(), plan["planes"], M, N, ldo, split_stride, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("c", BLOCKED_CASES, ids=[c["name"] for c in BLOCKED_CASES])
def test_tc_gemm_blocked_exact(tc, c):
    errs = run_blocked_case(c, *tc)
    assert not errs, "\n".join(errs)


# ---------------------------------------------------------------------------------------------------------------
# the logistic gradient through b2h_potential_and_grad
# ---------------------------------------------------------------------------------------------------------------
G_K, U_K = 6.0, 4.0


def _segment_rows(c):
    """fp32 accumulation lengths of the path: data rows per G segment, rows per fp32 potential partial sum."""
    path = logistic_path(c["mode"], c["dim"])
    if path == "two_kernel":
        lp = logreg_tc_plan(c["C"], c["N"], c["dim"])
        nv = lp["chunks"][0]
        g_rows = tc_plan(c["C"], c["dim"], nv, 3, lp["nsplit"], a_blocked=True)["kb_per"] * BK
        rp = tc_plan(c["C"], nv, c["dim"], 3, 1)
        u_rows = 32 * min(max(rp["per"], 1), rp["tiles_n"])
        return min(g_rows, nv), u_rows
    fp = fused_plan(c["C"], c["N"])
    return min(fp["per_cta"], fp["tiles_n"]) * FN, min(fp["per_cta"], fp["tiles_n"]) * 16


def reference_and_tolerance(X, y, q, inv_prior_var, fp16, n_seg, u_rows, chunk=2048):
    """float64 gradient and potential (GPU, chunks of chains) and the error model of the tensor-core paths.

    Per chain c and coordinate j, with r = sigmoid(s) - y:
      a_cj = sqrt(sum_n (x_nj r_cn)^2)     random errors in r_n and fp32 rounding of the sums grow with it
      b_j = sqrt(sum_n x_nj^2)             the approximate sigmoid (ex2 / rcp approximations): 2^-22 per residual
      e_cj = sqrt(sum_n x_nj^2 l_cn^2)     l_cn = sqrt(sum_k (x_nk q_ck)^2): error in s from the beta pieces and the
                                           fp32 sum over the dimension, 2^-23 l (fp16 x 2 carries 22 bits: 2^-21 l)
      E_cj = 2^-22 b_j + w 2^-23 e_cj + 2^-24 sqrt(n_seg) a_cj + 2^-25 n_acc (|g_cj| + a_cj)
             + 2^-23 (|g_cj| + |q_cj| / sigma^2),
    n_seg = data rows one fp32 accumulator sums (a CTA segment of the fused kernels, a split-K slice of the two-kernel
    product) and n_acc = n_seg pieces / 16 the accumulations into it (one per 16-deep MMA and piece).  The tensor
    cores' fp32 accumulation truncates (test_tc_fp32_accumulation_truncates pins it): each accumulation loses up to an
    ulp of the partial sum, and the partial sums grow towards g (steadily) and wander with a (randomly), hence the
    fourth term.  At the c5 shape it dominates: on a B200 (1000 W) the error of the 1 % largest |g| is 0.57 (median) to
    0.66 (max) times 2^-25 n_acc |g|, about 2e-4 |g|, so there a lost low piece (about 2^-12 a for fp16 x 2) hides
    under the kernel's own drift; the short-segment and exact cases catch it.  The last term is the float output.
    Tolerance G_K E.  The exact cases ("int_q0", "pieces") have tolerance 0: every operation in them is exact.
    Potential: E_U = 2^-21 N + w 2^-23 sqrt(sum_n r_n^2 l_n^2) + 2^-24 mean|u| L sqrt(N / 48) + 2^-23 |U|, the third
    term being a random walk of fp32 partial sums of L terms each (16 or 32 terms per addition); tolerance U_K E_U."""
    n_acc = n_seg * (2 if fp16 else 3) / 16
    dev = torch.device("cuda")
    Xd = torch.as_tensor(X, dtype=torch.float64, device=dev)
    X2 = Xd * Xd
    yd = torch.as_tensor(y, dtype=torch.float64, device=dev)
    w = 4.0 if fp16 else 1.0
    bj = X2.sum(0).sqrt()
    N = Xd.shape[0]
    G, E, U, EU = [], [], [], []
    for c0 in range(0, q.shape[0], chunk):
        qc = torch.as_tensor(q[c0:c0 + chunk], dtype=torch.float64, device=dev)
        S = qc @ Xd.T
        r = torch.sigmoid(S) - yd
        g = r @ Xd + inv_prior_var * qc
        l2 = (qc * qc) @ X2.T
        a = ((r * r) @ X2).sqrt()
        e = (l2 @ X2).sqrt()
        Eg = (2.0 ** -22 * bj + w * 2.0 ** -23 * e + 2.0 ** -24 * math.sqrt(n_seg) * a
              + 2.0 ** -25 * n_acc * (g.abs() + a) + 2.0 ** -23 * (g.abs() + inv_prior_var * qc.abs()))
        uterm = torch.logaddexp(torch.zeros_like(S), S) - yd * S
        Uc = uterm.sum(1) + 0.5 * inv_prior_var * (qc * qc).sum(1)
        Eu = (2.0 ** -21 * N + w * 2.0 ** -23 * (r * r * l2).sum(1).sqrt()
              + 2.0 ** -24 * uterm.abs().mean(1) * u_rows * math.sqrt(N / 48) + 2.0 ** -23 * Uc.abs())
        G.append(g)
        E.append(Eg)
        U.append(Uc)
        EU.append(Eu)
        del S, r, l2, a, e, uterm
    return torch.cat(G), torch.cat(E), torch.cat(U), torch.cat(EU)


def _problem(c, rng):
    """vals "pieces": an exact case in which every low piece carries weight.  Row n of X holds three entries +-1 in
    columns of its own, so every column has one non-zero.  Each chain's beta has, in those three columns, values with 21
    or 22 significant bits (granularity 2^-23) that cancel: s = 0 exactly whatever the summation order, yet the third
    bf16 piece (or the low fp16 piece) of each is non-zero and s != 0 without it.  y = 1/2 - t with t a float of 22
    significant bits in [1/4, 1/2), so r = sigmoid(0) - y = t exactly, and its low pieces are non-zero too.  Every fp32
    partial sum holds a multiple of 2^-24 below 1 (fp16 x 2: of 2^-9 below 2^14), which is exact, so the gradient
    g = X^T t + beta must come out bit for bit: a dropped or zeroed low piece of beta or of r changes it."""
    N, d, Cn = c["N"], c["dim"], c["C"]
    if c["vals"] == "pieces":
        assert 3 * N <= d
        cols = rng.permutation(d)[:3 * N].reshape(N, 3)
        sg = rng.choice([-1.0, 1.0], size=(N, 3))
        X = np.zeros((N, d))
        X[np.arange(N)[:, None], cols] = sg
        y = 0.5 - rng.integers(2 ** 21, 2 ** 22, N) * 2.0 ** -23
        q = np.zeros((Cn, d))
        vw = rng.integers(2 ** 20, 2 ** 21, size=(Cn, N, 2)) * 2.0 ** -23 * rng.choice([-1.0, 1.0], size=(Cn, N, 2))
        q[:, cols[:, 0]] = vw[:, :, 0]
        q[:, cols[:, 1]] = vw[:, :, 1]
        q[:, cols[:, 2]] = -(sg[:, 0] * vw[:, :, 0] + sg[:, 1] * vw[:, :, 1]) * sg[:, 2]
        return X, y, q
    if c["vals"] == "int_q0":
        X = _ints(rng, (N, d), 4)
        q = np.zeros((Cn, d))
        y = (rng.random(N) < 0.5).astype(np.float64)
        return X, y, q
    X = torch.tensor(rng.standard_normal((N, d)), dtype=torch.float32).bfloat16().double().numpy()
    beta = rng.standard_normal(d) / np.sqrt(d)
    if c["vals"] == "wrong_labels":
        # every chain near 2 beta, every label the opposite of its prediction: |r| close to 1, so a dropped low
        # residual or beta piece stands out against the approximate sigmoid
        y = (X @ beta < 0).astype(np.float64)
        return X, y, 2 * beta + 0.01 * rng.standard_normal((Cn, d))
    y = (rng.random(N) < 1 / (1 + np.exp(-X @ beta))).astype(np.float64)
    q = 0.3 * rng.standard_normal((Cn, d)) / np.sqrt(d / 16)
    return X, y, q


def _call_potential(lib, ctx, model, q, dtype, misaligned=False):
    """b2h_potential_and_grad with a workspace of 0xFF bytes (NaN as bf16, fp32 and fp64) and NaN-filled U and g.
    misaligned: q and g sit 4 bytes past a 16-byte boundary."""
    from aehmc_b200 import backend
    Cn, d = q.shape
    m = model.struct()
    code = backend.code(dtype)
    nbytes = lib.b2h_potential_workspace_bytes(C.byref(m), code, C.c_int64(Cn))
    ws = torch.full((nbytes,), 255, dtype=torch.uint8, device="cuda")
    off = 1 if misaligned else 0
    qb = torch.zeros(Cn * d + 4, dtype=dtype, device="cuda")
    qb[off:off + Cn * d] = torch.as_tensor(q, dtype=dtype).reshape(-1)
    gb = torch.full((Cn * d + 4,), float("nan"), dtype=dtype, device="cuda")
    U = torch.full((Cn,), float("nan"), dtype=dtype, device="cuda")
    esz = qb.element_size()
    vp = C.c_void_p
    rc = lib.b2h_potential_and_grad(ctx, C.byref(m), C.c_int(code), vp(qb.data_ptr() + off * esz), vp(U.data_ptr()),
                                    vp(gb.data_ptr() + off * esz), C.c_int64(Cn), vp(ws.data_ptr()), C.c_int64(nbytes))
    torch.cuda.synchronize()
    if rc != 0:
        raise AssertionError(f"b2h_potential_and_grad returned {rc}: {lib.b2h_last_error()}")
    return U, gb[off:off + Cn * d].view(Cn, d)


def run_fused_case(c, lib, ctx):
    import aehmc_b200 as ab
    dtype = torch.float64 if c["dtype"] == "f64" else torch.float32
    rng = np.random.default_rng(zlib.crc32(c["name"].encode()))
    X, y, q = _problem(c, rng)
    flag = {"fp16x2": True, "bf16x3": "bf16x3", "two_kernel": "two_kernel"}[c["mode"]]
    model = ab.models.LogisticRegression(X, y, 1.0, dtype=dtype, tensor_core=flag)
    want = {"fp16x2": 4.0, "bf16x3": 2.0, "two_kernel": 3.0}[c["mode"]]
    tag = c["name"]
    if model.tc_flag != want:
        return [f"{tag}: model flag {model.tc_flag}, the case needs {want}"]
    qd = torch.as_tensor(q, dtype=dtype).double().numpy()             # what the kernel sees
    U, g = _call_potential(lib, ctx, model, qd, dtype)
    n_seg, u_rows = _segment_rows(c)
    return compare(tag, X, y, qd, U, g, c["mode"] == "fp16x2", n_seg, u_rows,
                   exact=c["vals"] in ("int_q0", "pieces"), recheck=(lib, ctx, model, dtype) if c["misaligned"] else None)


def compare(tag, X, y, qd, U, g, fp16, n_seg, u_rows, exact=False, recheck=None):
    errs = []
    if not (torch.isfinite(g).all() and torch.isfinite(U).all()):
        return [f"{tag}: NaN or inf in the result (an unwritten workspace slot was read)"]
    g_ref, Eg, U_ref, EU = reference_and_tolerance(X, y, qd, 1.0, fp16, n_seg, u_rows)
    err = (g.double() - g_ref).abs()
    # a coordinate no data row touches has E = 0 and must come out exact (0 / 0 counts as 0, x / 0 as inf)
    rel = torch.where(err > 0, err / Eg, torch.zeros_like(err))
    urel = (U.double() - U_ref).abs() / EU
    ratio = float(rel.max()) / G_K
    uratio = float(urel.max()) / U_K
    RATIOS[tag] = (ratio, uratio)
    # how much of the error the truncation drift 2^-25 n_acc |g| explains, on the 1 % largest |g|
    ga = g_ref.abs().flatten()
    top = ga >= ga.kthvalue(max(1, int(0.99 * ga.numel()))).values
    drift = (err.flatten() / (2.0 ** -25 * n_seg * (2 if fp16 else 3) / 16 * g_ref.abs().flatten()))[top]
    print(f"{tag}: gradient error / tolerance {ratio:.4f}, potential {uratio:.4f} (max |dU| "
          f"{float((U.double() - U_ref).abs().max()):.3e}); error / truncation drift on the largest |g|: median "
          f"{float(drift.median()):.3f}, max {float(drift.max()):.3f}")
    if exact and not torch.equal(g.double(), g_ref):
        n = int((g.double() != g_ref).sum())
        errs.append(f"{tag}: exact case: {n} gradient elements differ from the exact gradient, max {float(err.max()):.3e}")
    if ratio > 1.0:
        i = int(rel.argmax())
        ci, j = divmod(i, g.shape[1])
        errs.append(f"{tag}: gradient error {float(err.view(-1)[i]):.3e} at chain {ci}, coordinate {j}: "
                    f"{ratio:.2f} x the tolerance {G_K * float(Eg.view(-1)[i]):.3e}")
    if uratio > 1.0:
        i = int(urel.argmax())
        errs.append(f"{tag}: potential error {float((U.double() - U_ref).abs()[i]):.3e} at chain {i}: {uratio:.2f} x "
                    f"the tolerance {U_K * float(EU[i]):.3e}")
    if recheck is not None:
        lib, ctx, model, dtype = recheck
        U2, g2 = _call_potential(lib, ctx, model, qd, dtype, misaligned=True)
        if not torch.equal(g2, g):
            errs.append(f"{tag}: misaligned q / g: {int((g2 != g).sum())} gradient elements differ from the aligned call")
        du = (U2.double() - U.double()).abs()
        ubound = 2.0 ** -22 * (U.double().abs() + 0.5 * float((torch.as_tensor(qd) ** 2).sum(1).max()))
        if not bool((du <= ubound).all()):
            errs.append(f"{tag}: misaligned q / g: potential differs by {float(du.max()):.3e} from the aligned call")
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("c", FUSED_CASES, ids=[c["name"] for c in FUSED_CASES])
def test_logistic_gradient_paths(tc, c):
    errs = run_fused_case(c, *tc)
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
def test_tc_fp32_accumulation_truncates(tc):
    """The gradient tolerance assumes that the tensor cores' fp32 accumulation truncates (rounds towards zero).  With
    the accumulator at 2^24 (ulp 2) each further k-block adds 1.5: rounding to nearest would give 2^24 + 2 per block,
    truncation leaves 2^24."""
    lib, ctx = tc
    K = 8 * BK
    b = np.zeros((8, K))
    b[:, 0] = 2.0 ** 24
    for blk in range(1, 8):
        b[:, blk * BK], b[:, blk * BK + 1] = 1.0, 0.5
    A = _bf16_bits(np.ones((1, K))).cuda()
    B = _bf16_bits(b).cuda()
    out = torch.full((8,), SENTINEL, dtype=torch.float32, device="cuda")
    assert lib.b2h_tc_gemm_bf16(ctx, A.data_ptr(), K, B.data_ptr(), K, out.data_ptr(), 1, 8, K, 1, 1, 8, 1, 8) == 0
    torch.cuda.synchronize()
    got = out.double().cpu().numpy()
    print(f"accumulation of 2^24 + 7 x 1.5: {got[0] - 2.0 ** 24:+.1f} over 2^24")
    assert np.all(got == 2.0 ** 24), got - 2.0 ** 24


@pytest.mark.gpu
def test_c5_shape_every_chain(tc):
    """131072 chains on the c5 data (N = 100000, D = 128), fp16 x 2, FP32 state: about 7 chain-tile segments per CTA,
    two partial planes per chain tile.  Every chain's gradient and potential against the float64 reference.  Measured on
    a B200 (1000 W): gradient 0.16 of its tolerance, potential 0.27 (largest |U error| 0.12, at U of order 1e4)."""
    import bench
    import aehmc_b200 as ab
    lib, ctx = tc
    X, y, imm = bench.make_logistic_problem(100000, 128)
    Cn = 131072
    q = bench.initial_positions("logistic", Cn, 128) + np.sqrt(imm) * np.random.default_rng(9).standard_normal((Cn, 128))
    model = ab.models.LogisticRegression(X, y, 1.0, dtype=torch.float32, tensor_core=True)
    assert model.tc_flag == 4.0
    qd = q.astype(np.float32).astype(np.float64)
    U, g = _call_potential(lib, ctx, model, qd, torch.float32)
    fp = fused_plan(Cn, 100000)
    c = dict(mode="fp16x2", dim=128, C=Cn, N=100000)
    errs = compare("c5-shape", X, y, qd, U, g, True, *_segment_rows(c))
    assert fp["planes"] == 2
    assert not errs, "\n".join(errs)
