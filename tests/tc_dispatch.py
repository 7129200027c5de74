"""Host dispatch of the tcgen05 kernels (csrc/tc_gemm.cu, csrc/logreg.cu) restated in Python: which kernel a launch
runs, how many split-K planes it writes and how the fused kernels cut their work.  Shared by the tensor-core tests."""
SMS = 148
BM = BN = 128
BK = 64
FN = 64
RES_A_BLOCKS, RES_KB = 6, 2
CHUNK_BYTES = 256 << 20


def cdiv(a, b):
    return -(-a // b)


def tc_plan(M, N, K, pieces, nsplit, a_blocked=False):
    """tc_launch: split clamping and the resident / persistent choice."""
    kb_total = cdiv(K, BK)
    ns = min(max(nsplit, 1), kb_total)
    kb_per = cdiv(kb_total, ns)
    ns = cdiv(kb_total, kb_per)
    tiles_n, tiles_m = cdiv(N, BN), cdiv(M, BM)
    total = tiles_n * tiles_m * ns
    p = dict(kb_total=kb_total, kb_per=kb_per, planes=ns, tiles_m=tiles_m, tiles_n=tiles_n, total=total)
    if not a_blocked and ns == 1 and pieces * kb_total <= RES_A_BLOCKS and kb_total <= RES_KB and total >= 2 * SMS:
        per = cdiv(total, SMS)
        grid = cdiv(total, per)
        cross = any((b * per) // tiles_n != (min(total, (b + 1) * per) - 1) // tiles_n for b in range(grid))
        p.update(kernel="resident", per=per, grid=grid, crosses_row_tile=cross)
    else:
        grid = min(total, SMS)
        p.update(kernel="persistent", per=0, grid=grid, max_tiles_per_cta=cdiv(total, grid))
    return p


def logreg_tc_plan(C_, N, d):
    """plan_logreg_tc: data rows per chunk and split-K slices of the second product."""
    nc = (2 * CHUNK_BYTES) // (C_ * 6)
    nc = max(128, (nc // 128) * 128)
    if nc > N:
        nc = cdiv(N, 128) * 128
    tiles = cdiv(C_, 128) * cdiv(d, 128)
    ns = max(1, min(cdiv(296, tiles), cdiv(nc, 512)))
    chunks = [min(nc, N - n0) for n0 in range(0, N, nc)]
    return dict(n_chunk=nc, nsplit=ns, chunks=chunks)


def fused_plan(C_, N):
    """tc_logistic_fused*: items (chain tile, 64 data rows) per CTA; logistic_fused_planes."""
    tiles_m, tiles_n = cdiv(C_, BM), cdiv(N, FN)
    total = tiles_m * tiles_n
    per = cdiv(total, SMS)
    grid = cdiv(total, per)
    on_tile = any((b * per) % tiles_n == 0 for b in range(1, grid))
    return dict(tiles_m=tiles_m, tiles_n=tiles_n, per_cta=per, grid=grid, planes=cdiv(tiles_n, per) + 1,
                boundary_on_chain_tile=on_tile)


def logistic_path(mode, dim):
    if mode == "fp16x2" and dim <= 128:
        return "fused16"
    if mode == "bf16x3" and dim <= 128:
        return "fused"
    return "two_kernel"
