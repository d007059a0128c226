"""Kernel 2's column top-2 variant (mv_k2_sim_top2_cols_ld) against fp64 torch on the same rounded operands, and against
the top-2 kernel it shares everything else with: row outputs and the packed column arg-max bit-identical."""
from ctypes import c_size_t

import pytest
import torch

pytestmark = pytest.mark.gpu

DTYPES = {"bf16": (torch.bfloat16, 0), "tf32": (None, 1), "f16": (torch.float16, 2)}


def round_operand(x, dtype):
    if dtype == "bf16":
        return x.to(torch.bfloat16).float()
    if dtype == "f16":
        return x.to(torch.float16).float()
    bits = x.contiguous().view(torch.int32)  # tf32-exact: 10 explicit mantissa bits
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def _operands(A, B, dtype):
    t16 = DTYPES[dtype][0]
    Ad = A.cuda().to(t16).contiguous() if t16 else A.cuda().contiguous()
    Bd = B.cuda().to(t16).contiguous() if t16 else B.cuda().contiguous()
    return Ad, Bd


def run_cols(mv, A, B, dtype, cluster, n_live=None, m_live=None):
    """(row_val, row_idx, col_val, col_idx, col_best) of mv_k2_sim_top2_cols_ld, on the host."""
    L = mv._lib
    n, C = A.shape
    m = B.shape[0]
    dev = torch.device("cuda")
    Ad, Bd = _operands(A, B, dtype)
    row_val = torch.full((n, 2), 7.0, device=dev)
    row_idx = torch.full((n, 2), -9, dtype=torch.int32, device=dev)
    col_val = torch.full((m, 2), 7.0, device=dev)
    col_idx = torch.full((m, 2), -9, dtype=torch.int32, device=dev)
    col_best = torch.full((m,), 5, dtype=torch.int64, device=dev)
    ws_bytes = L.load().mv_k2_cols_workspace_bytes(n, m)
    ws = torch.full((ws_bytes,), 0xAB, dtype=torch.uint8, device=dev)  # stale records must never be read
    nd = torch.tensor([n_live], dtype=torch.int32, device=dev) if n_live is not None else None
    md = torch.tensor([m_live], dtype=torch.int32, device=dev) if m_live is not None else None
    L.call("mv_k2_sim_top2_cols_ld", L.ptr(Ad), C, L.ptr(Bd), C, n, m, C, L.ptr(nd), L.ptr(md), DTYPES[dtype][1], cluster,
           L.ptr(row_val), L.ptr(row_idx), L.ptr(col_val), L.ptr(col_idx), L.ptr(col_best), L.ptr(ws), c_size_t(ws_bytes),
           mv.correspondence._stream())
    torch.cuda.synchronize()
    return row_val.cpu(), row_idx.cpu(), col_val.cpu(), col_idx.cpu(), col_best.cpu()


def run_top2(mv, A, B, dtype, cluster, n_live=None, m_live=None):
    """(row_val, row_idx, col_best) of mv_k2_sim_top2_ld on the same operands."""
    L = mv._lib
    n, C = A.shape
    m = B.shape[0]
    dev = torch.device("cuda")
    Ad, Bd = _operands(A, B, dtype)
    row_val = torch.empty((n, 2), device=dev)
    row_idx = torch.empty((n, 2), dtype=torch.int32, device=dev)
    col_best = torch.empty((m,), dtype=torch.int64, device=dev)
    ws_bytes = L.load().mv_k2_workspace_bytes(n, m)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    nd = torch.tensor([n_live], dtype=torch.int32, device=dev) if n_live is not None else None
    md = torch.tensor([m_live], dtype=torch.int32, device=dev) if m_live is not None else None
    L.call("mv_k2_sim_top2_ld", L.ptr(Ad), C, L.ptr(Bd), C, n, m, C, L.ptr(nd), L.ptr(md), DTYPES[dtype][1], cluster,
           L.ptr(row_val), L.ptr(row_idx), L.ptr(col_best), L.ptr(ws), c_size_t(ws_bytes), mv.correspondence._stream())
    torch.cuda.synchronize()
    return row_val.cpu(), row_idx.cpu(), col_best.cpu()


def check_cols(S, cv, ci, nl, ml, m):
    """column top-2 of S (nl, ml) fp64 against the kernel's (m, 2) outputs."""
    tol = 1e-4 * max(1.0, float(S.abs().max()))
    k = min(2, nl)
    val, idx = torch.topk(S.t(), k, dim=1)
    assert (cv[:ml, :k].double() - val).abs().max() <= tol
    srt = torch.sort(S, dim=0, descending=True).values
    clear1 = (srt[0] - srt[1] > 2 * tol) if nl > 1 else torch.ones(ml, dtype=torch.bool)
    assert torch.equal(ci[:ml, 0].long()[clear1], idx[:, 0][clear1])
    if nl > 2:
        clear2 = clear1 & (srt[1] - srt[2] > 2 * tol)
        assert torch.equal(ci[:ml, 1].long()[clear2], idx[:, 1][clear2])
    # whichever rows were returned own the returned values, and the two are distinct rows
    got = S.t().gather(1, ci[:ml, :k].long().clamp(min=0))
    assert (got - cv[:ml, :k].double()).abs().max() <= tol
    if nl > 1:
        assert (ci[:ml, 0] != ci[:ml, 1]).all()
    else:
        assert (ci[:ml, 1] == -1).all() and (cv[:ml, 1] < -1e38).all()
    if ml < m:
        assert (ci[ml:] == -1).all() and (cv[ml:] < -1e38).all()


def check(mv, n, m, C, dtype, cluster, seed=0, n_live=None, m_live=None):
    g = torch.Generator().manual_seed(7000 * n + m + C + seed)
    A = round_operand(torch.randn(n, C, generator=g), dtype)
    B = round_operand(torch.randn(m, C, generator=g), dtype)
    rv, ri, cv, ci, cb = run_cols(mv, A, B, dtype, cluster, n_live, m_live)
    rv2, ri2, cb2 = run_top2(mv, A, B, dtype, cluster, n_live, m_live)
    # the rows and the packed arg-max are the top-2 kernel's, bit for bit
    assert torch.equal(rv.view(torch.int32), rv2.view(torch.int32)) and torch.equal(ri, ri2)
    assert torch.equal(cb, cb2)
    nl = n if n_live is None else n_live
    ml = m if m_live is None else m_live
    S = A[:nl].double() @ B[:ml].double().t()
    check_cols(S, cv, ci, nl, ml, m)
    # col_best decodes to the first column candidate
    live = ci[:, 0] >= 0
    assert torch.equal((0xFFFFFFFF - (cb[live] & 0xFFFFFFFF)).int(), ci[live, 0])
    assert (cb[~live] == 0).all()


# the tile-edge shapes of test_gpu_k2.py; K extents ending inside a 128-byte row exercise the partial last k-block
SHAPES = [
    (1, 1, 8), (1, 2, 8), (5, 3, 16), (128, 256, 64), (129, 257, 64), (300, 280, 64), (127, 255, 72),
    (700, 1500, 128), (1000, 777, 768), (2048, 2048, 256), (196, 20, 768), (20, 196, 768), (260, 300, 776), (150, 520, 104),
]


@pytest.mark.parametrize("n,m,C", SHAPES)
@pytest.mark.parametrize("dtype", ["bf16", "tf32", "f16"])
@pytest.mark.parametrize("cluster", [0, 2, 4, 20])  # 20 = MV_CLUSTER_PAIR (cta_group::2)
def test_k2_cols_against_fp64(mv, n, m, C, dtype, cluster):
    check(mv, n, m, C, dtype, cluster)


@pytest.mark.parametrize("cluster", [0, 2, 4, 20])
def test_k2_cols_device_resident_counts(mv, cluster):
    check(mv, 900, 1100, 64, "bf16", cluster, n_live=611, m_live=1023)
    check(mv, 900, 1100, 64, "tf32", cluster, n_live=1, m_live=2)
    check(mv, 700, 300, 72, "f16", cluster, n_live=257, m_live=1)


@pytest.mark.parametrize("cluster", [0, 20])
def test_k2_cols_exact_ties_go_to_the_lower_row(mv, cluster):
    g = torch.Generator().manual_seed(3)
    B = round_operand(torch.randn(300, 64, generator=g), "bf16")
    A = round_operand(torch.randn(400, 64, generator=g), "bf16")
    A[137] = A[5]    # duplicated query rows: the same similarity to every column
    A[300] = A[5]
    A[260] = B[11] * 4  # column 11's best, duplicated below in row 391
    A[391] = A[260]
    rv, ri, cv, ci, cb = run_cols(mv, A, B, "bf16", cluster)
    assert ci[11, 0] == 260 and ci[11, 1] == 391 and cv[11, 0] == cv[11, 1]
    for j in range(300):
        if ci[j, 0] in (5, 137, 300):
            assert ci[j, 0] == 5 and ci[j, 1] == 137
    # every similarity equal: the two lowest rows everywhere
    rv, ri, cv, ci, cb = run_cols(mv, torch.ones(260, 64), torch.ones(600, 64), "bf16", cluster)
    assert (ci[:, 0] == 0).all() and (ci[:, 1] == 1).all() and (cv == 64).all()


def test_k2_cols_repeatable(mv):
    g = torch.Generator().manual_seed(5)
    A = torch.randn(1500, 128, generator=g)
    B = torch.randn(1300, 128, generator=g)
    for cluster in (0, 2, 4, 20):
        a = run_cols(mv, A, B, "bf16", cluster)
        b = run_cols(mv, A, B, "bf16", cluster)
        assert all(torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x, y.view(torch.int32) if y.dtype == torch.float32 else y)
                   for x, y in zip(a, b))


@pytest.mark.parametrize("cluster", [-1, 20])
def test_k2_cols_self_product_full_size(mv, cluster):
    """19200^2 x 768 with B = A: every column's best row is the column itself and its second the true runner-up."""
    g = torch.Generator(device="cuda").manual_seed(11)
    n, C = 19200, 768
    X = torch.nn.functional.normalize(torch.randn(n, C, device="cuda", generator=g), dim=1).to(torch.bfloat16)
    L = mv._lib
    dev = X.device
    row_val, row_idx = torch.empty((n, 2), device=dev), torch.empty((n, 2), dtype=torch.int32, device=dev)
    col_val, col_idx = torch.empty((n, 2), device=dev), torch.empty((n, 2), dtype=torch.int32, device=dev)
    col_best = torch.empty((n,), dtype=torch.int64, device=dev)
    ws_bytes = L.load().mv_k2_cols_workspace_bytes(n, n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    L.call("mv_k2_sim_top2_cols_ld", L.ptr(X), C, L.ptr(X), C, n, n, C, None, None, L.MV_DTYPE_BF16, cluster, L.ptr(row_val),
           L.ptr(row_idx), L.ptr(col_val), L.ptr(col_idx), L.ptr(col_best), L.ptr(ws), c_size_t(ws_bytes),
           mv.correspondence._stream())
    torch.cuda.synchronize()
    ar = torch.arange(n, device=dev, dtype=torch.int32)
    assert torch.equal(col_idx[:, 0], ar)
    # the runner-up by fp32 products of the bf16 rows, in blocks; ties within accumulation noise are excused
    Xf = X.float()
    for r0 in range(0, n, 2048):
        S = Xf @ Xf[r0:r0 + 2048].t()  # (n, block): column j of the block
        S[r0 + torch.arange(S.shape[1], device=dev), torch.arange(S.shape[1], device=dev)] = -2.0
        top = torch.topk(S, 2, dim=0)
        got = col_idx[r0:r0 + 2048, 1].long()
        gap = top.values[0] - top.values[1]
        ok = (got == top.indices[0]) | (gap < 1e-4)
        assert bool(ok.all()), int((~ok).sum())
        assert (col_val[r0:r0 + 2048, 1] - top.values[0]).abs().max() < 1e-4
