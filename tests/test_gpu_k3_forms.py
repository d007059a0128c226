"""Kernel 3's ratio / mutual step in every row form against fp64, and the tf32c operand planes of kernel 1.

Kernel 3 (csrc/k3_score.cu k3_ratio_mutual_kernel; csrc/lr_gram.cu lr_k3_ratio_mutual_kernel) turns kernel 2's two proposed
neighbours of a query into fp32 distances, their order, the ratio weight and the mutual flag.  It is tested on its own here:
the candidates are handed in (a third of them in the wrong order) and the reference is fp64 1 - cos of the fp32 rows kernel
1 wrote in the same launch as the row planes kernel 3 reads (the oracle's interpolated rows for the Gram-matrix form).
The tf32c planes (mv_k1_sample_tf32c) are checked bit for bit, and kernel 2 on them against the fp64 product a . b."""
from ctypes import c_size_t

import pytest
import torch
import torch.nn.functional as F

from oracle import restated
from test_gpu_f16c import collinear_rows

pytestmark = pytest.mark.gpu

FORMS = ("fp32", "split", "f16c")
SENT_D, SENT_W, SENT_MU = -7.0, -9.0, 0xAB  # what rows past the live count must still hold afterwards


def k1_rows(mv, form, X, role, mu):
    """kernel 1 in MV_SAMPLE_ROWS mode (normalising) with the roles of the dense helpers (_pair_maps: the query rows carry
    dotvec = mu, the target rows are stored relative to center = mu): (the planes kernel 3 reads, the fp32 rows of the
    same launch)."""
    L, C_ = mv._lib, mv.correspondence
    Xd = X.cuda().contiguous()
    n, C = Xd.shape
    f32 = torch.empty((n, C), device="cuda")
    if form == "fp32":
        L.call("mv_k1_sample_normalize", L.MV_SAMPLE_ROWS, L.ptr(Xd), C, 0, 0, None, None, n, 1, None, None, L.ptr(f32), None,
               C_._stream())
        planes = (f32,)
    elif form == "split":
        hi = torch.empty((n, C), dtype=torch.bfloat16, device="cuda")
        lo = torch.empty_like(hi)
        L.call("mv_k1_sample_normalize", L.MV_SAMPLE_ROWS, L.ptr(Xd), C, 0, 0, None, None, n, 1, L.ptr(hi), L.ptr(lo), L.ptr(f32),
               None, C_._stream())
        planes = (hi, lo)
    else:
        hi = torch.empty((n, L.f16c_pitch(C)), dtype=torch.float16, device="cuda")
        lo = torch.empty((n, C), dtype=torch.float16, device="cuda")
        center, dotvec = (mu, None) if role == L.MV_ROLE_TARGET else (None, mu)
        L.call("mv_k1_sample_f16c", L.MV_SAMPLE_ROWS, L.ptr(Xd), C, 0, 0, None, None, n, 1, role, L.ptr(center), L.ptr(dotvec), None,
               L.ptr(hi), hi.shape[1], L.ptr(lo), L.ptr(f32), None, None, C_._stream())
        planes = (hi, lo)
    torch.cuda.synchronize()
    return planes, f32


def outputs(n, given):
    """fresh outputs filled with sentinels, and a device copy of the candidates"""
    return (given.to(torch.int32).cuda().contiguous(), torch.full((n, 2), SENT_D, device="cuda"), torch.full((n,), SENT_W, device="cuda"),
            torch.full((n,), SENT_MU, dtype=torch.uint8, device="cuda"))


def run_k3(mv, form, A, B, C, mu, given, n_dev=None, col_best=None, ratio_test=1, with_outputs=True):
    """one kernel-3 launch of the given row form: (row_idx, dists, weight, mutual) on the host"""
    L, C_ = mv._lib, mv.correspondence
    ridx, d, w, mu8 = outputs(given.shape[0], given)
    if not with_outputs:
        d = w = mu8 = col_best = None
    tail = (L.ptr(n_dev), given.shape[0], L.ptr(ridx), L.ptr(col_best), int(ratio_test), L.ptr(d), L.ptr(w), L.ptr(mu8), C_._stream())
    if form == "fp32":
        L.call("mv_k3_ratio_mutual", L.ptr(A[0]), L.ptr(B[0]), C, *tail)
    elif form == "split":
        L.call("mv_k3_ratio_mutual_split", L.ptr(A[0]), L.ptr(A[1]), L.ptr(B[0]), L.ptr(B[1]), C, *tail)
    else:
        L.call("mv_k3_ratio_mutual_f16c", L.ptr(A[0]), L.ptr(A[1]), L.ptr(B[0]), L.ptr(B[1]), C, A[0].shape[1], L.ptr(mu), *tail)
    torch.cuda.synchronize()
    return tuple(None if t is None else t.cpu() for t in (ridx, d, w, mu8))


def dist64(X, Y, idx):
    """fp64 1 - cos(X[i], Y[idx[i, k]]) with F.cosine_similarity's clamp of each norm at 1e-8 (a zero row gives 1); 2 for a
    missing candidate (-1)"""
    X, Y, idx = X.double().cpu(), Y.double().cpu(), idx.long()
    j = idx.clamp(min=0)
    cos = (X[:, None, :] * Y[j]).sum(-1) / (X.norm(dim=1).clamp(min=1e-8)[:, None] * Y.norm(dim=1).clamp(min=1e-8)[j])
    return torch.where(idx >= 0, 1 - cos, torch.full_like(cos, 2.0))


def cos64(X, Y):
    Xn = F.normalize(X.double().cpu(), dim=1)
    Yn = F.normalize(Y.double().cpu(), dim=1)
    return Xn @ Yn.t()


def col_best_of(S):
    """col_best as kernel 2 packs it (order bits above, 0xffffffff - row below) for the fp64 column arg-max"""
    return ((1 << 32) | (0xFFFFFFFF - S.argmax(0))).to(torch.int64)


def check_rows(given, got, d, w, mu8, X, Y, col_best, ratio_test, live, tol=1e-6):
    """what every form owes its live rows: the candidates handed in, re-ranked; distances within tol of fp64; the fp64 order
    wherever the fp64 gap exceeds 1e-6 and ties to the lower index; the weight of the kernel's own distances; the mutual flag
    decoded from col_best.  Rows past the live count keep their sentinels."""
    g, r = given[:live].long(), got[:live].long()
    assert torch.equal(r.sort(1).values, g.sort(1).values)
    dl = d[:live]
    d64 = dist64(X[:live], Y, r)
    err = (dl.double() - d64).abs()
    assert float(err.max()) <= tol, (float(err.max()), int(err.flatten().argmax()) // 2)
    clear = (d64[:, 0] - d64[:, 1]).abs() > 1e-6
    assert bool((d64[clear, 0] < d64[clear, 1]).all())
    assert bool((dl[:, 0] <= dl[:, 1]).all())
    tie = (dl[:, 0] == dl[:, 1]) & (r[:, 1] >= 0)
    assert bool((r[tie, 0] < r[tie, 1]).all())
    if ratio_test:
        torch.testing.assert_close(w[:live], restated.ratio_weights(dl), rtol=0, atol=1e-7)
    else:
        assert torch.equal(w[:live], dl[:, 0])
    j0 = r[:, 0]
    want = torch.zeros(live, dtype=torch.bool)
    if col_best is not None:
        pk = col_best.cpu()[j0.clamp(min=0)]
        want = (j0 >= 0) & (pk != 0) & ((0xFFFFFFFF - (pk & 0xFFFFFFFF)) == torch.arange(live))
    assert torch.equal(mu8[:live], want.to(torch.uint8))
    assert torch.equal(got[live:], given[live:].to(torch.int32))
    assert bool((d[live:] == SENT_D).all()) and bool((w[live:] == SENT_W).all()) and bool((mu8[live:] == SENT_MU).all())


def candidates(S, swap_every=3):
    """the fp64 top-2 of every row, a third of the pairs handed in swapped"""
    idx = torch.topk(S, 2, dim=1).indices
    idx[::swap_every] = idx[::swap_every].flip(1)
    return idx


@pytest.mark.parametrize("C", [8, 200, 768, 2048, 3072])
@pytest.mark.parametrize("kind", ["iid", "collinear"])
@pytest.mark.parametrize("form", FORMS)
def test_row_forms_against_fp64(mv, form, kind, C):
    """k3_score.cu:96-218 (k3_ratio_mutual_kernel, the fp32 / split / f16c row loads at :113-164 and the tail at :182-217)
    against fp64 1 - cos of kernel 1's own fp32 rows: distances to 1e-6, the fp64 order, weights from the kernel's distances
    (ratio_test 1 and 0), the mutual flag of the col_best passed in."""
    n, m = 257, 301
    g = torch.Generator().manual_seed(C)
    if kind == "iid":
        X, Y = 3.0 * torch.randn(n, C, generator=g), torch.randn(m, C, generator=g)
    else:
        X, Y = collinear_rows(n, C, 20 + C) * 3.0, collinear_rows(m, C, 21 + C)
    mu = mv.correspondence._center(Y.cuda().contiguous(), m)
    A, A32 = k1_rows(mv, form, X, mv._lib.MV_ROLE_QUERY, mu)
    B, B32 = k1_rows(mv, form, Y, mv._lib.MV_ROLE_TARGET, mu)
    S = cos64(A32, B32)
    given = candidates(S)
    cb = col_best_of(S).cuda()
    # split rows carry 16 mantissa bits (hi + lo to 2^-17 per element); their independent roundings average out over the
    # channels to well below 1e-6, except over 8 of them: measured 2.1e-6 at C = 8
    tol = 5e-6 if (form, C) == ("split", 8) else 1e-6
    for ratio_test in (1, 0):
        got, d, w, mu8 = run_k3(mv, form, A, B, C, mu, given, col_best=cb, ratio_test=ratio_test)
        check_rows(given, got, d, w, mu8, A32, B32, cb, ratio_test, n, tol)
    assert int(mu8.sum()) > 0  # the mutual branch is exercised


def edge_candidates(S, n, m, dup, zero_t):
    """candidates with every branch of the tail: row 0 (j, -1), row 1 (-1, -1), row 2 the duplicated target row pair handed
    in as (j', j), rows 3 / 4 the zero target row first / second; rows from n // 2 on hold valid sentinel indices"""
    given = candidates(S)
    given[0, 1] = -1
    given[1] = -1
    given[2] = torch.tensor([dup[1], dup[0]])
    given[3] = torch.tensor([zero_t, (zero_t + 11) % m])
    given[4] = torch.tensor([(zero_t + 13) % m, zero_t])
    given[n // 2:] = torch.tensor([m - 1, 0])
    return given


def check_edges(given, got, d, w, mu8, dup, ratio_test):
    assert got[0].tolist() == given[0].tolist() and float(d[0, 1]) == 2.0           # j1 = -1: MISSING_DIST, no swap
    assert got[1].tolist() == [-1, -1] and d[1].tolist() == [2.0, 2.0] and int(mu8[1]) == 0
    assert float(w[1]) == (0.0 if ratio_test else 2.0)
    assert got[2].tolist() == [dup[0], dup[1]] and float(d[2, 0]) == float(d[2, 1])  # bit-equal distances: the lower index


@pytest.mark.parametrize("C", [200, 2048])
@pytest.mark.parametrize("form", FORMS)
def test_row_forms_edge_cases(mv, form, C):
    """the branches of k3_score.cu's tail on every row form: the device-side live count (:103, rows past it untouched), a
    missing candidate (MISSING_DIST, :193-194), bit-equal distances (the lower index wins, :195), an empty col_best column
    (:210-216), a zero query row and a zero target row (distance 1 as F.cosine_similarity gives, COS_EPS at :192-194; the
    f16c target row is stored relative to the centre and its rebuild residual counts as zero, :183-190), and null outputs
    (row_idx re-ranked exactly as with every output)."""
    n, m = 96, 80
    X, Y = collinear_rows(n, C, 31) * 2.0, collinear_rows(m, C, 32)
    zero_q, zero_t, dup = 5, 7, (20, 40)
    X[zero_q] = 0.0
    Y[zero_t] = 0.0
    Y[dup[1]] = Y[dup[0]]
    mu = mv.correspondence._center(Y.cuda().contiguous(), m)
    A, A32 = k1_rows(mv, form, X, mv._lib.MV_ROLE_QUERY, mu)
    B, B32 = k1_rows(mv, form, Y, mv._lib.MV_ROLE_TARGET, mu)
    assert torch.equal(B32[dup[0]], B32[dup[1]])
    S = cos64(A32, B32)
    given = edge_candidates(S, n, m, dup, zero_t)
    given[zero_q] = torch.tensor([10, 3])
    cb = col_best_of(S)
    empty = int(given[6].max())
    cb[empty] = 0
    cb[int(given[8, 0])] = (1 << 32) | (0xFFFFFFFF - 8)  # row 8's first candidate names it back: mutual unless re-ranked
    cb = cb.cuda()
    live = n // 2
    n_dev = torch.tensor([live], dtype=torch.int32, device="cuda")
    for ratio_test in (1, 0):
        got, d, w, mu8 = run_k3(mv, form, A, B, C, mu, given, n_dev=n_dev, col_best=cb, ratio_test=ratio_test)
        check_rows(given, got, d, w, mu8, A32, B32, cb, ratio_test, live)
        check_edges(given, got, d, w, mu8, dup, ratio_test)
        assert got[zero_q].tolist() == [3, 10] and d[zero_q].tolist() == [1.0, 1.0]
        for i in (3, 4):
            k = got[i].tolist().index(zero_t)
            assert abs(float(d[i, k]) - 1.0) <= 1e-6, (i, float(d[i, k]))
        assert int(mu8[6]) == 0 or int(got[6, 0]) != empty
    nulls = run_k3(mv, form, A, B, C, mu, given, n_dev=n_dev, with_outputs=False)[0]
    assert torch.equal(nulls, got)


def lr_pair(mv, syn, kind):
    """a pair prepared for the exact low-rank route (no kernel 1), its target image with a duplicated point, the oracle's
    interpolated rows, and the Gram matrix and inverse norms of mv_lr_gram_exact / the builders"""
    C_ = mv.correspondence
    dev = torch.device("cuda")
    if kind == "depth":
        p = syn.scannet_pair(6, C=256, h=15, w=20, H=60, W=80)
        Kh, Kinv = C_._host_mat(p["K"]), C_._host_mat(p["K"].inverse())
        s0 = C_.prepare_depth_side(p["feat_0"].cuda(), p["depth_0"], Kh, Kinv, dev, want_rows=False)
        s1 = C_.prepare_depth_side(p["feat_1"].cuda(), p["depth_1"], Kh, Kinv, dev, want_rows=False)
        f0 = restated.depth_side(p["feat_0"], p["depth_0"], p["K"])[1]
        f1 = restated.depth_side(p["feat_1"], p["depth_1"], p["K"])[1]
    else:  # the disc reaches the map border: bicubic taps clamped onto the same source pixel
        p = syn.navi_pair(6, C=256, h=14, w=14, H=48, W=48, radius=30.0)
        s0 = C_.prepare_xyz_side(p["feat_0"].cuda(), p["xyz_grid_0"], dev, want_rows=False)
        s1 = C_.prepare_xyz_side(p["feat_1"].cuda(), p["xyz_grid_1"], dev, want_rows=False)
        f0 = restated.xyz_side(p["feat_0"], p["xyz_grid_0"])[1]
        f1 = restated.xyz_side(p["feat_1"], p["xyz_grid_1"])[1]
    n, m = s0.n, s1.n
    assert (n, m) == (f0.shape[0], f1.shape[0])
    dup = (10, m - 5)
    s1.coords[dup[1]] = s1.coords[dup[0]]
    f1 = f1.clone()
    f1[dup[1]] = f1[dup[0]]
    x = C_._lowrank_operands(s0, s1, n, m, None, None, exact=True)[3]
    torch.cuda.synchronize()
    return s0, s1, f0, f1, x, dup


@pytest.mark.parametrize("kind", ["depth", "xyz"])
def test_gram_form_against_fp64(mv, syn, kind):
    """mv_k3_ratio_mutual_lr (lr_gram.cu:420-483) on the Gram matrix of mv_lr_gram_exact and the builders' inverse norms,
    bilinear (taps partly off the map, dropped) and bicubic (clamped taps repeating a source pixel): every row's distances
    within 1e-6 of fp64 1 - cos of the oracle's interpolated rows, candidates from the fp64 top-2 (a third swapped); a
    duplicated target point (an exact tie: the lower index, :460), missing candidates (:437-439), the device-side live count
    (:425), the mutual flag and an empty column (:475-481), and null outputs."""
    L, C_ = mv._lib, mv.correspondence
    s0, s1, f0, f1, x, dup = lr_pair(mv, syn, kind)
    n, m = s0.n, s1.n
    C, h, w = s0.fshape
    c = s0.coords.cpu()[:n]
    fx, fy = c[:, 0].floor(), c[:, 1].floor()
    if kind == "depth":
        assert bool(((fx < 0) | (fx + 1 > w - 1) | (fy < 0) | (fy + 1 > h - 1)).any())
    else:
        assert bool(((fx - 1 < 0) | (fx + 2 > w - 1) | (fy - 1 < 0) | (fy + 2 > h - 1)).any())
    S = cos64(f0, f1)
    cb = col_best_of(S)
    cb[int(candidates(S)[6].max())] = 0
    cb = cb.cuda()

    def run(given, n_dev=None, ratio_test=1, with_outputs=True):
        ridx, d, wt, mu8 = outputs(n, given)
        if not with_outputs:
            d = wt = mu8 = None
        L.call("mv_k3_ratio_mutual_lr", s0.mode, L.ptr(s0.coords), L.ptr(s1.coords), L.ptr(x["inv0"]), L.ptr(x["inv1"]), L.ptr(x["G"]),
               x["ld"], 0, x["off_t"], h, w, L.ptr(n_dev), n, L.ptr(ridx), L.ptr(cb if with_outputs else None), ratio_test, L.ptr(d),
               L.ptr(wt), L.ptr(mu8), C_._stream())
        torch.cuda.synchronize()
        return tuple(None if t is None else t.cpu() for t in (ridx, d, wt, mu8))

    given = candidates(S)
    for ratio_test in (1, 0):
        got, d, wt, mu8 = run(given, ratio_test=ratio_test)
        check_rows(given, got, d, wt, mu8, f0, f1, cb, ratio_test, n)
    assert int(mu8.sum()) > n // 4
    edges = edge_candidates(S, n, m, dup, 0)
    live = n // 2
    n_dev = torch.tensor([live], dtype=torch.int32, device="cuda")
    for ratio_test in (1, 0):
        got, d, wt, mu8 = run(edges, n_dev=n_dev, ratio_test=ratio_test)
        check_rows(edges, got, d, wt, mu8, f0, f1, cb, ratio_test, live)
        check_edges(edges, got, d, wt, mu8, dup, ratio_test)
    assert torch.equal(run(edges, n_dev=n_dev, with_outputs=False)[0], got)


def tf32_rn(x):
    """round to nearest tf32, ties away from zero, as a bit operation on the fp32 pattern: (bits + 0x1000) & 0xffffe000"""
    b = x.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    b = (b + 0x1000) & 0xFFFFE000
    return torch.where(b >= 1 << 31, b - (1 << 32), b).to(torch.int32).view(torch.float32)


def tf32c_rows(mv, X, role, mu, pitch=None, fill=9.0):
    """mv_k1_sample_tf32c in MV_SAMPLE_ROWS mode with the helpers' roles: (operand plane (n, pitch), fp32 rows)"""
    L, C_ = mv._lib, mv.correspondence
    Xd = X.cuda().contiguous()
    n, C = Xd.shape
    pitch = pitch or L.tf32c_pitch(C)
    op = torch.full((n, pitch), fill, device="cuda")
    f32 = torch.empty((n, C), device="cuda")
    center, dotvec = (mu, None) if role == L.MV_ROLE_TARGET else (None, mu)
    L.call("mv_k1_sample_tf32c", L.MV_SAMPLE_ROWS, L.ptr(Xd), C, 0, 0, None, None, n, 1, role, L.ptr(center), L.ptr(dotvec), None,
           L.ptr(op), pitch, L.ptr(f32), None, C_._stream())
    torch.cuda.synchronize()
    return op, f32


@pytest.mark.parametrize("C", [768, 2048, 3072, 200])  # 200: the generic (any C) instantiation
def test_tf32c_row_planes_bit_exact(mv, C):
    """k1_sample.cu:425-438 and :480-491 (put / put_aug with out_op32): the plane is tf32_rn(out_f32 - mu) for targets and
    tf32_rn(out_f32) for queries, bit for bit against a CPU emulation of tf32_rn (:373) on the kernel's own fp32 rows; the
    augmentation columns are (1, 1, 1, 0...) for targets and, for queries, three tf32-exact pieces p0 = tf32_rn(r),
    p1 = tf32_rn(r - p0), p2 = r - p0 - p1 of one fp32 r within 2e-6 of fp64 row . mu; a padded pitch is never written past C + 8."""
    L = mv._lib
    n = 300
    X = collinear_rows(n, C, 1) * 3.0  # not unit: kernel 1 normalises
    mu = mv.correspondence._center(X.cuda().contiguous(), n)
    pitch = L.tf32c_pitch(C) + 32
    for role in (L.MV_ROLE_TARGET, L.MV_ROLE_QUERY):
        op, f32 = tf32c_rows(mv, X, role, mu, pitch)
        op, f32 = op.cpu(), f32.cpu()
        y = f32 - mu.cpu()[None] if role == L.MV_ROLE_TARGET else f32
        assert torch.equal(op[:, :C].view(torch.int32), tf32_rn(y).view(torch.int32))
        assert bool((op[:, C + 8:] == 9.0).all())
        aug = op[:, C:C + 8]
        if role == L.MV_ROLE_TARGET:
            assert torch.equal(aug, torch.tensor([1.0, 1.0, 1.0, 0, 0, 0, 0, 0]).expand(n, 8))
            continue
        assert bool((aug[:, 3:] == 0).all())
        p = aug[:, :3]
        assert torch.equal(tf32_rn(p), p)
        r = p.double().sum(1)
        assert torch.equal(r.float().double(), r)  # the three pieces add up to one fp32 number exactly
        r = r.float()
        assert torch.equal(p[:, 0], tf32_rn(r)) and torch.equal(p[:, 1], tf32_rn(r - p[:, 0]))
        want_r = (f32.double() * mu.cpu().double()[None]).sum(1)
        assert float((r.double() - want_r).abs().max()) <= 2e-6


@pytest.mark.parametrize("C,cluster", [(768, -1), (2048, -1), (2048, 0), (3072, 20), (264, 2)])
def test_tf32c_product_is_the_uncentred_product(mv, C, cluster):
    """kernel 2 (MV_DTYPE_TF32, C + 8 columns) on tf32c planes, every cluster form: row values / indices and column arg-max
    of a . b (not a . (b - mu)) on nearly collinear rows, the bound of the f16c form's test."""
    L, C_ = mv._lib, mv.correspondence
    n, m = 700, 900
    X, Y = collinear_rows(n, C, 2), collinear_rows(m, C, 3)
    mu = C_._center(Y.cuda().contiguous(), m)
    A, _ = tf32c_rows(mv, X, L.MV_ROLE_QUERY, mu)
    B, _ = tf32c_rows(mv, Y, L.MV_ROLE_TARGET, mu)
    row_val = torch.empty((n, 2), device="cuda")
    row_idx = torch.empty((n, 2), dtype=torch.int32, device="cuda")
    col_best = torch.empty(m, dtype=torch.int64, device="cuda")
    wsb = L.load().mv_k2_workspace_bytes(n, m)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    L.call("mv_k2_sim_top2_ld", L.ptr(A), A.shape[1], L.ptr(B), B.shape[1], n, m, C + 8, None, None, L.MV_DTYPE_TF32, cluster,
           L.ptr(row_val), L.ptr(row_idx), L.ptr(col_best), L.ptr(ws), c_size_t(wsb), C_._stream())
    col_val = torch.empty(m, device="cuda")
    col_idx = torch.empty(m, dtype=torch.int32, device="cuda")
    L.call("mv_k2_unpack_col", L.ptr(col_best), m, L.ptr(col_val), L.ptr(col_idx), C_._stream())
    torch.cuda.synchronize()
    S = F.normalize(X.double(), dim=1) @ F.normalize(Y.double(), dim=1).t()
    val, idx = torch.topk(S, 3, dim=1)
    assert (row_val.cpu().double() - val[:, :2]).abs().max() < 4e-5
    clear = (val[:, 0] - val[:, 1]) > 5e-5
    assert clear.float().mean() > 0.5
    assert torch.equal(row_idx.cpu().long()[clear, 0], idx[clear, 0])
    clear2 = clear & ((val[:, 1] - val[:, 2]) > 5e-5)
    assert torch.equal(row_idx.cpu().long()[clear2, 1], idx[clear2, 1])
    cs = torch.topk(S, 2, dim=0)
    cclear = (cs.values[0] - cs.values[1]) > 5e-5
    assert torch.equal(col_idx.cpu().long()[cclear], cs.indices[0][cclear])
    assert (col_val.cpu().double() - cs.values[0]).abs().max() < 4e-5
