"""Drop-in for the reference's ``evals/utils/correspondence.py`` backed by libmvmatch.so (sm_100a).

Same function names, argument meaning and return tuples as the reference module
(/root/reference/evals/utils/correspondence.py, cited per function below); the arithmetic runs in
three hand-written CUDA kernels reached through the C ABI of include/mvmatch.h:

    kernel 1  sample / upsample + L2-normalise            (csrc/k1_sample.cu)
    kernel 2  tcgen05 similarity GEMM + row top-2 / column arg-max   (csrc/k2_sim.cu)
    kernel 3  fp32 distance recompute, ratio test, mutual check, top-k, scoring   (csrc/k3_score.cu)

Inputs may live on the CPU (NAVI / ScanNet callers, evaluate_navi_correspondence.py:149-150,
render_scannet_correspondence.py:201) or on a CUDA device (SPair caller); results come back on the
device of the first feature argument, indices as int64, like the reference.  There is no CPU
implementation here: without a CUDA device every compute entry point raises.
"""
import os
from ctypes import c_float, c_int, c_size_t, c_void_p

import numpy as np
import torch

from . import _lib as L

__all__ = [
    "faiss_knn", "knn_points", "get_correspondences_ratio_test", "calculate_ratio_test", "get_topk_matches",
    "get_grid", "grid_to_pointcloud", "sample_pointcloud_features", "argmax_2d", "project_3dto2d", "error_auc",
    "estimate_correspondence_depth", "estimate_correspondence_xyz", "compute_binned_performance",
    "set_match_precision", "match_rows", "prepare_depth_side", "prepare_xyz_side", "MatchResult",
]

# operand type of kernel 2:
#   "f16"  (default) tcgen05 kind::f16 on fp16 "f16c" rows: target rows stored relative to a centre, the query rows carry
#          their dot product with that centre in three extra columns (include/mvmatch.h, mv_k1_sample_f16c).  Same tensor
#          rate as bf16 with the ranking precision of fp32 on real backbone features (CNN maps are nearly collinear:
#          a plain bf16 product ranks the wrong neighbour there, DESIGN.md section 4)
#   "bf16" tcgen05 kind::f16 on plain bf16 rows     "tf32" kind::tf32 on fp32 rows (half the rate)
# cluster = B-tile multicast width
DEFAULT_DTYPE = "f16"
_CFG = {
    "dtype": os.environ.get("MVMATCH_DTYPE", DEFAULT_DTYPE),
    "cluster": int(os.environ.get("MVMATCH_CLUSTER", "-1")),  # -1 = let the library choose (MV_CLUSTER_AUTO)
    # host-tensor calls of the two dense helpers replay a CUDA graph cached per input shape (0 = launch eagerly)
    "helper_graphs": int(os.environ.get("MVMATCH_HELPER_GRAPHS", "1")),
    # how kernel 1 hands the fp32 rows to kernel 3 on the bf16 path: "split" = bf16 hi + bf16 residual planes
    # (4 bytes / element, hi doubles as kernel 2's operand), "f32" = bf16 + fp32 rows (6 bytes / element)
    "rows": os.environ.get("MVMATCH_ROWS", "split"),
    # 1 = the NAVI-style side through the tiled cluster kernel (csrc/k1_grid.cu) where its shape is covered.  Measured on
    # B200 (bench.py --k1-only, same box): 56.2 us against 32.3 us of the point-run kernel for a NAVI-shaped side -- a third
    # of the L2 traffic, but 16 warps per SM behind a cluster barrier per round are latency-bound -- so it is OFF by default
    "k1_grid": int(os.environ.get("MVMATCH_K1_GRID", "0")),
    # host-tensor calls of the dense helpers: two graphs (target side / the rest) so that the second image's upload overlaps
    # the first one's kernels (evaluation.GraphedPairMatcher.load_and_replay_split); 0 = one graph after both uploads
    "helper_split": int(os.environ.get("MVMATCH_HELPER_SPLIT", "1")),
    # kernel 2's product over the SOURCE PIXELS of the target image instead of the channels (csrc/lr_gram.cu, "low-rank
    # proposal"): "auto" = where it pays (dense helpers, fp16 operands, h*w + 8 <= C / 5 and a large similarity matrix: the
    # ScanNet-shaped pairs, 312 instead of 2056 columns), "1" = wherever it applies, "0" = never
    "lowrank": os.environ.get("MVMATCH_LOWRANK", "auto"),
    # with the low-rank proposal: 1 = kernel 3's two distances per query also come from the (exact, CUDA-core fp32) Gram matrix
    # of the source pixels (mv_lr_gram_exact + mv_k3_ratio_mutual_lr) and the interpolated rows are never materialised
    # (no kernel 1); 0 = kernel 1 writes the row planes and kernel 3 reads them, as for the dense product
    "lowrank_k3": os.environ.get("MVMATCH_LOWRANK_K3", "1"),
}
_HELPER_GRAPHS = {}  # (kind, shapes, num_corr, ratio_test, dtype, cluster, K bytes) -> evaluation.GraphedPairMatcher
_HELPER_GRAPHS_MAX = 12


# bench.py sets _PROFILE["k2_events"] = [] to collect (start, end, flop) CUDA-event records of kernel 2
_PROFILE = {}


def set_match_precision(dtype=None, cluster=None, helper_graphs=None, rows=None, k1_grid=None, lowrank=None, lowrank_k3=None):
    """Choose kernel 2's operand type ("f16" | "bf16" | "tf32"), its cluster width (1, 2 or 4), whether the dense
    helpers replay cached CUDA graphs for host-tensor calls, and the row format between kernels 1 and 3
    ("split" | "f32", see _CFG)."""
    if k1_grid is not None:
        _CFG["k1_grid"] = int(bool(k1_grid))
    if lowrank is not None:
        if str(lowrank) not in ("auto", "0", "1"):
            raise ValueError("lowrank must be 'auto', 0 or 1")
        _CFG["lowrank"] = str(lowrank)
    if lowrank_k3 is not None:
        _CFG["lowrank_k3"] = "1" if int(lowrank_k3) else "0"
    if rows is not None:
        if rows not in ("split", "f32"):
            raise ValueError("rows must be 'split' or 'f32'")
        _CFG["rows"] = rows
    if helper_graphs is not None:
        _CFG["helper_graphs"] = int(bool(helper_graphs))
    if dtype is not None:
        if dtype not in ("f16", "bf16", "tf32"):
            raise ValueError("dtype must be 'f16', 'bf16' or 'tf32'")
        _CFG["dtype"] = dtype
    if cluster is not None:
        if cluster not in (-1, 1, 2, 4, 20):
            raise ValueError("cluster must be -1 (auto), 1, 2, 4 (B-tile multicast width) or 20 (CTA pairs, cta_group::2)")
        _CFG["cluster"] = cluster
    return dict(_CFG)


# ------------------------------------------------------------------------------------------------
# plumbing
# ------------------------------------------------------------------------------------------------
def _device():
    if not torch.cuda.is_available():
        raise RuntimeError("mvmatch has no CPU path: a CUDA (sm_100a) device is required")
    return torch.device("cuda", torch.cuda.current_device())


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()


def _empty(shape, dtype, dev):
    return torch.empty(shape, dtype=dtype, device=dev)


def _hwc(feat, prenorm=False):
    """(C, h, w) fp32 device map -> channel-last (h*w, C); prenorm = F.normalize(feat, dim=channel)."""
    C, h, w = feat.shape
    out = _empty((h * w, C), torch.float32, feat.device)
    scratch = _empty((h * w,), torch.float32, feat.device) if prenorm else None
    L.call("mv_chw_to_hwc", L.ptr(feat), L.ptr(out), C, h * w, int(prenorm), L.ptr(scratch), _stream())
    return out


_FEAT_DTYPES = {torch.float32: L.MV_FEAT_F32, torch.bfloat16: L.MV_FEAT_BF16, torch.float16: L.MV_FEAT_F16}


def _is_channel_last(feat):
    """True when a (C, h, w) tensor is a permuted view of contiguous (h, w, C) memory -- the layout ViT tokens
    have before tokens_to_output's .contiguous() (evals/models/utils.py:111-114) and channels_last CNN outputs."""
    C, h, w = feat.shape
    return feat.dtype in _FEAT_DTYPES and feat.stride() == (1, w * C, C) and not (h * w == 1 or C == 1)


def _feature_map(feat, dev, prenorm=False):
    """(C, h, w) features (any device) -> (channel-last (h*w, C) fp32 device map, C, h, w).

    A channel-last view is used as it is (no copy, no transpose kernel); the reference's contiguous (C, h, w)
    layout goes through mv_chw_to_hwc.  prenorm always runs the kernel (it rescales every pixel)."""
    C, h, w = feat.shape
    _check_C(C)
    if feat.dtype in (torch.bfloat16, torch.float16) and not prenorm:
        # autocast backbones: upload the 16-bit map as it is (half the bytes) and widen on the device (exact)
        cl = _is_channel_last(feat)
        f = feat.detach().to(device=dev, non_blocking=True)
        f = f if (cl and _is_channel_last(f)) else f.contiguous()
        out = _empty((h * w, C), torch.float32, dev)
        L.call("mv_feat_to_hwc_f32", L.ptr(f), _FEAT_DTYPES[feat.dtype], int(cl), C, h * w, L.ptr(out), _stream())
        return out, C, h, w
    if _is_channel_last(feat) and not prenorm:
        f = feat.detach().to(device=dev, non_blocking=True)
        if _is_channel_last(f):
            return f.permute(1, 2, 0).reshape(h * w, C), C, h, w
    return _hwc(_f32(feat, dev), prenorm), C, h, w


def _check_C(C):
    if C % 8 != 0:
        raise ValueError(f"feature dimension {C} must be a multiple of 8 for the tensor-core path")


def _sample(mode, src, C, h, w, coords, n_dev, n_max, normalize, want_bf16, want_f32, taps=None, want_lo=False,
            role=L.MV_ROLE_QUERY, center=None, dotvec=None, pixdot=None):
    """kernel 1.  src: (h*w, C) channel-last (or (n, C) rows for MV_SAMPLE_ROWS).
    Returns (16-bit rows, fp32 rows, 16-bit residual rows); the ones not asked for are None.
    The 16-bit rows are bf16 (n, C) for the "bf16" operand type and fp16 "f16c" rows (n, f16c_pitch(C)) for "f16":
    role / center / dotvec are the f16c parameters of mv_k1_sample_f16c."""
    dev = src.device
    if _CFG["dtype"] == "tf32" and want_f32 and (center is not None or dotvec is not None or pixdot is not None):
        # tf32c: exact fp32 rows for kernel 3 + a centred, tf32-rounded operand plane with the augmentation columns for
        # kernel 2 (returned in the operand-rows slot)
        o32 = _empty((max(n_max, 1), C), torch.float32, dev)
        oop = _empty((max(n_max, 1), L.tf32c_pitch(C)), torch.float32, dev)
        if n_max > 0:
            L.call("mv_k1_sample_tf32c", mode, L.ptr(src), C, h, w, L.ptr(coords), L.ptr(n_dev), n_max, int(normalize), role,
                   L.ptr(center), L.ptr(dotvec), L.ptr(pixdot), L.ptr(oop), oop.shape[1], L.ptr(o32), L.ptr(taps), _stream())
        return oop, o32, None
    f16 = _CFG["dtype"] == "f16" and (want_bf16 or want_lo)
    t16 = torch.float16 if f16 else torch.bfloat16
    o16 = _empty((max(n_max, 1), L.f16c_pitch(C) if f16 else C), t16, dev) if (want_bf16 or want_lo) else None
    olo = _empty((max(n_max, 1), C), t16, dev) if want_lo else None
    o32 = _empty((max(n_max, 1), C), torch.float32, dev) if want_f32 else None
    if n_max > 0 and f16:
        L.call("mv_k1_sample_f16c", mode, L.ptr(src), C, h, w, L.ptr(coords), L.ptr(n_dev), n_max, int(normalize), role,
               L.ptr(center), L.ptr(dotvec), L.ptr(pixdot), L.ptr(o16), o16.shape[1], L.ptr(olo), L.ptr(o32), None, L.ptr(taps),
               _stream())
    elif n_max > 0:
        L.call("mv_k1_sample_normalize", mode, L.ptr(src), C, h, w, L.ptr(coords), L.ptr(n_dev), n_max, int(normalize),
               L.ptr(o16), L.ptr(olo), L.ptr(o32), L.ptr(taps), _stream())
    return o16, o32, olo


def _center(rows, n, n_dev=None, step=1):
    """(C,) fp32 centre of the L2-normalised rows (mean direction of every step-th row): mv_rows_center."""
    C = rows.shape[1]
    mu = _empty((C,), torch.float32, rows.device)
    scratch = _empty(((n + step - 1) // step,), torch.float32, rows.device)
    L.call("mv_rows_center", L.ptr(rows), C, n, L.ptr(n_dev), step, L.ptr(scratch), L.ptr(mu), _stream())
    return mu


def _row_format(rows=None):
    """(want 16-bit rows, want fp32 rows, want 16-bit residual rows) of kernel 1 for the configured kernel-2 operand
    type and row format."""
    if _CFG["dtype"] == "tf32":
        return False, True, False
    if (rows or _CFG["rows"]) == "split":
        return True, False, True
    return True, True, False


class MatchResult:
    """Device-side outputs of one directional match (kernels 2 + 3)."""

    __slots__ = ("k", "k_dev", "sel_src", "sel_dst", "sel_weight", "mutual", "row_idx", "dists", "weight", "col_best")


def _k2_operands(A16, A32, B16, B32, C):
    """kernel 2's operands for prepared rows of C channels under the configured operand type: (A, B, columns of the
    product, MV_DTYPE_*).  The 16-bit rows, or the centred tf32c planes, which ride in the same slot; plain fp32 rows
    for tf32 without them.  f16c / tf32c rows add their 8 augmentation columns to the product."""
    tf32 = _CFG["dtype"] == "tf32"
    f16 = _CFG["dtype"] == "f16"
    tf32c = tf32 and A16 is not None and B16 is not None
    A, B = (A16, B16) if (not tf32 or tf32c) else (A32, B32)
    Ck = C + 8 if (f16 or tf32c) else C
    return A, B, Ck, L.MV_DTYPE_TF32 if tf32 else (L.MV_DTYPE_F16 if f16 else L.MV_DTYPE_BF16)


def match_rows(A16, A32, B16, B32, n, m, num_corr, ratio_test=True, n_dev=None, m_dev=None, want_topk=True, run_k3=True,
               A_lo=None, B_lo=None, center_B=None, C=None, proposal=None):
    """kernel 2 + kernel 3 on prepared rows.

    A16/B16: (n, C)/(m, C) bf16 rows or (n, pitch)/(m, pitch) fp16 f16c rows (query / target role; None when the
    tf32 path is selected), A32/B32: fp32 rows -- or None when the split form is used: A_lo/B_lo are then the 16-bit
    residual planes of A16/B16.  center_B: the centre f16c target rows are relative to (None: not centred).
    Mirrors get_correspondences_ratio_test (correspondence.py:63-102, bidirectional=False):
    2-NN -> fp32 cosine distances -> ratio weights -> top-num_corr, plus the mutual-NN flag.
    n, m are the live counts when n_dev/m_dev are None, otherwise upper bounds.
    proposal: (A_op, B_op, K) fp16 operand rows of _lowrank_operands -- kernel 2 then ranks their product over K columns
    (the same cosine similarities in the basis of the source pixels) while kernel 3 still reads the exact rows.
    """
    ref = A32 if A32 is not None else A16
    dev = ref.device
    tf32 = _CFG["dtype"] == "tf32"
    f16 = _CFG["dtype"] == "f16"
    C = ref.shape[1] if A32 is not None else (C if C is not None else ref.shape[1])
    split = A32 is None or B32 is None
    if split and (tf32 or A_lo is None or B_lo is None or A16 is None or B16 is None):
        raise ValueError("split rows need a 16-bit operand type and both residual planes")
    st = _stream()
    res = MatchResult()
    row_val = _empty((n, 2), torch.float32, dev)
    row_idx = _empty((n, 2), torch.int32, dev)
    col_best = _empty((m,), torch.int64, dev)
    lib = L.load()
    ws_bytes = lib.mv_k2_workspace_bytes(n, m)
    ws = _empty((ws_bytes,), torch.uint8, dev)
    if split:
        C = A_lo.shape[1]
    k2_A, k2_B, Ck, k2_dtype = _k2_operands(A16, A32, B16, B32, C)
    ld = k2_A.shape[1]
    if proposal is not None:
        k2_A, k2_B, Ck = proposal
        k2_dtype = L.MV_DTYPE_F16
    prof = _PROFILE.get("k2_events")
    if prof is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    L.call("mv_k2_sim_top2_ld", L.ptr(k2_A), k2_A.shape[1], L.ptr(k2_B), k2_B.shape[1], n, m, Ck, L.ptr(n_dev), L.ptr(m_dev),
           k2_dtype, _CFG["cluster"], L.ptr(row_val),
           L.ptr(row_idx), L.ptr(col_best), L.ptr(ws), c_size_t(ws_bytes), st)
    if prof is not None:
        ev1.record()
        prof.append((ev0, ev1, (n, m, Ck, n_dev, m_dev)))
    res.row_idx, res.col_best = row_idx, col_best
    if not run_k3:  # raw kernel-2 neighbours (inner-product order), no cosine re-ranking
        return res
    dists = _empty((n, 2), torch.float32, dev)
    weight = _empty((n,), torch.float32, dev)
    mutual = _empty((n,), torch.uint8, dev)
    if split and f16:
        L.call("mv_k3_ratio_mutual_f16c", L.ptr(A16), L.ptr(A_lo), L.ptr(B16), L.ptr(B_lo), C, ld, L.ptr(center_B), L.ptr(n_dev), n,
               L.ptr(row_idx), L.ptr(col_best), int(ratio_test), L.ptr(dists), L.ptr(weight), L.ptr(mutual), st)
    elif split:
        L.call("mv_k3_ratio_mutual_split", L.ptr(A16), L.ptr(A_lo), L.ptr(B16), L.ptr(B_lo), C, L.ptr(n_dev), n,
               L.ptr(row_idx), L.ptr(col_best), int(ratio_test), L.ptr(dists), L.ptr(weight), L.ptr(mutual), st)
    else:
        L.call("mv_k3_ratio_mutual", L.ptr(A32), L.ptr(B32), C, L.ptr(n_dev), n, L.ptr(row_idx), L.ptr(col_best),
               int(ratio_test), L.ptr(dists), L.ptr(weight), L.ptr(mutual), st)
    res.row_idx, res.dists, res.weight, res.mutual, res.col_best = row_idx, dists, weight, mutual, col_best
    if want_topk:
        k = min(int(num_corr), n)
        res.k = k
        res.sel_src = _empty((max(k, 1),), torch.int32, dev)
        res.sel_dst = _empty((max(k, 1),), torch.int32, dev)
        res.sel_weight = _empty((max(k, 1),), torch.float32, dev)
        res.k_dev = _empty((1,), torch.int32, dev)
        L.call("mv_k3_topk_matches", L.ptr(weight), L.ptr(row_idx), L.ptr(n_dev), n, k, L.ptr(res.sel_src),
               L.ptr(res.sel_dst), L.ptr(res.sel_weight), L.ptr(res.k_dev), st)
    return res


def _gather(src, idx, k, k_dev=None):
    """rows src[idx[:k]] through the library (src (n, width) fp32, idx int32); with k_dev only the first
    *k_dev (<= k) rows are gathered, the rest of the output is left as allocated."""
    width = src.shape[1]
    out = _empty((k, width), torch.float32, src.device)
    if k > 0:
        L.call("mv_gather_rows", L.ptr(src), width, L.ptr(idx), L.ptr(k_dev), k, L.ptr(out), _stream())
    return out


def _rows_from_features(F, normalize, dev, role=L.MV_ROLE_QUERY, center=None, dotvec=None):
    """(N, C) features -> (16-bit rows or None, fp32 rows), optionally L2-normalised (correspondence.py:47-48)."""
    F = _f32(F, dev)
    n, C = F.shape
    _check_C(C)
    want16 = _CFG["dtype"] != "tf32"
    if not normalize and not want16:
        return None, F
    return _sample(L.MV_SAMPLE_ROWS, F, C, 0, 0, None, None, n, normalize, want16, True, role=role, center=center,
                   dotvec=dotvec)[:2]


def _rows_pair(X_f, Y_f, dev):
    """query rows of X_f and target rows of Y_f for one cosine match: ((A16, A32), (B16, B32), centre of the targets)."""
    mu = None
    if _CFG["dtype"] != "bf16" and Y_f.shape[0] > 0:
        Y = _f32(Y_f, dev)
        mu = _center(Y, Y.shape[0], step=max(1, Y.shape[0] // 1024))  # any vector near the mean direction will do
        Y_f = Y
    return (_rows_from_features(X_f, True, dev, L.MV_ROLE_QUERY, dotvec=mu),
            _rows_from_features(Y_f, True, dev, L.MV_ROLE_TARGET, center=mu), mu)


# ------------------------------------------------------------------------------------------------
# reference interface: nearest neighbours
# ------------------------------------------------------------------------------------------------
def faiss_knn(query, target, k):
    """L2 k-NN: (squared L2 distances ascending, int64 indices).  correspondence.py:14-23.
    k <= 16 runs on kernel 2 wherever the target has at least k rows; larger k, and targets with fewer than k rows, take
    the exact blocked search of _exact_knn_blocks (which returns min(k, m) columns).

    Neighbours are PROPOSED at tf32 precision -- kernel 2's two best per row for k <= 2, its row top-KP epilogue
    (KP = 8 for k <= 6, 16 up to k = 16) otherwise -- and fp32 distances recomputed from the rows decide their order
    (mv_knn_rerank for k > 2).  Ranking tolerance: a neighbour whose squared distance is within ~1e-3 relative of the
    last candidate's can be missed (the north-star gap rule); missing neighbours (target smaller than k) come back as
    (-1, inf) like faiss.
    The search runs on kernel 2 through the identity ||q-t||^2 = ||q||^2 + ||t||^2 - 2 q.t : the rows are
    extended by (1, -||t||^2/2) split into tf32-exact pieces so that the inner-product order is the L2
    order; the returned distances are recomputed in fp32 for the winners.
    """
    dev = _device()
    in_dev = query.device
    q = _f32(query, dev)
    t = _f32(target, dev)
    n, C = q.shape
    m = t.shape[0]
    if k > 2:
        if not _fused_knn_applies(n, m, int(k)):
            d, idx = _exact_knn_blocks(q, t, int(k))
            return d.to(in_dev), idx.to(in_dev)
        qe, te = _l2_operands(q, t)
        cand = _topk_candidates(qe, te, n, m, qe.shape[1], L.MV_DTYPE_TF32, int(k))
        d, idx = _rerank(q, t, cand, int(k), L.MV_METRIC_L2SQ)
        return d.to(in_dev), idx.long().to(in_dev)
    if k < 1:
        raise ValueError("k must be positive")
    qe, te = _l2_operands(q, t)
    saved = dict(_CFG)
    try:
        _CFG["dtype"] = "tf32"
        r = match_rows(None, qe, None, te, n, m, 0, want_topk=False, run_k3=False)
    finally:
        _CFG.update(saved)
    # both candidates always: the tf32 product only PROPOSES them, their fp32 distances decide the order (so k = 1
    # also returns the better of the two); a missing neighbour (m < k) is faiss's (-1, inf), never a wrapped index
    idx = r.row_idx.long()
    have = idx >= 0
    d = ((q[:, None, :] - t[idx.clamp(min=0)]) ** 2).sum(dim=-1)
    d = torch.where(have, d, torch.full_like(d, float("inf")))
    swap = d[:, 1] < d[:, 0]
    d = torch.where(swap[:, None], d.flip(1), d)
    idx = torch.where(swap[:, None], idx.flip(1), idx)
    return d[:, :k].contiguous().to(in_dev), idx[:, :k].contiguous().to(in_dev)


def _l2_operands(q, t):
    """kernel 2's tf32 operands of an L2 search: (n, Cp) query rows and (m, Cp) target rows whose inner-product order along
    a row is the squared-L2 order."""
    dev = q.device
    n, C = q.shape
    m = t.shape[0]
    # extra columns: q' = [q, 1, 1, 1, 0..], t' = [t, h0, h1, h2, 0..] with h0+h1+h2 = -||t||^2/2, each piece
    # holding <= 10 mantissa bits so the tf32 tensor-core product does not round it
    half = -0.5 * (t * t).sum(dim=1)
    pieces = []
    rem = half.clone()
    for _ in range(3):
        mant, expo = torch.frexp(rem)
        p = torch.ldexp(torch.round(mant * 1024.0) / 1024.0, expo)
        pieces.append(p)
        rem = rem - p
    Cp = ((C + 3 + 7) // 8) * 8
    qe = torch.zeros((n, Cp), dtype=torch.float32, device=dev)
    te = torch.zeros((m, Cp), dtype=torch.float32, device=dev)
    # targets relative to their mean: q.(t - mu) differs from q.t by a per-query constant, so the order along a row is
    # unchanged while the tf32 rounding error shrinks with |t - mu| (the same idea as the f16c rows)
    qe[:, :C] = q
    qe[:, C:C + 3] = 1.0
    te[:, :C] = t - t.mean(dim=0, keepdim=True) if m > 1 else t
    for i, p in enumerate(pieces):
        te[:, C + i] = p
    return qe, te


_FUSED_K_MAX = 16  # longest row list of kernel 2's top-KP epilogue


def _fused_knn_applies(n, m, k):
    """whether k > 2 neighbours come from kernel 2's top-KP epilogue + the fp32 re-rank (else: _exact_knn_blocks)."""
    return 3 <= k <= _FUSED_K_MAX and n >= 1 and m >= k


def _topk_candidates(A, B, n, m, Ck, dtype, k):
    """kernel 2 with the row top-KP epilogue on operand rows A (n, pitch) / B (m, pitch) over Ck columns: (n, KP) int32
    candidate columns, best first.  KP = 8 for k <= 6, else 16: at least two spare candidates wherever the list allows."""
    kp = 8 if k <= 6 else 16
    dev = A.device
    row_val = _empty((n, kp), torch.float32, dev)
    row_idx = _empty((n, kp), torch.int32, dev)
    ws_bytes = L.load().mv_k2_topk_workspace_bytes(n, m, kp)
    ws = _empty((ws_bytes,), torch.uint8, dev)
    L.call("mv_k2_sim_topk_ld", L.ptr(A), A.shape[1], L.ptr(B), B.shape[1], n, m, Ck, None, None, dtype, _CFG["cluster"], kp,
           L.ptr(row_val), L.ptr(row_idx), L.ptr(ws), c_size_t(ws_bytes), _stream())
    return row_idx


def _rerank(Q, T, cand, k, metric):
    """fp32 distances of every query's candidates (mv_knn_rerank): the k nearest, ascending, ties to the lower index."""
    n, C = Q.shape
    dist = _empty((n, k), torch.float32, Q.device)
    idx = _empty((n, k), torch.int32, Q.device)
    L.call("mv_knn_rerank", L.ptr(Q), Q.stride(0), L.ptr(T), T.stride(0), C, None, n, L.ptr(cand), cand.shape[1], k, metric,
           L.ptr(dist), L.ptr(idx), _stream())
    return dist, idx


def _exact_knn_blocks(q, t, k):
    """exact fp32 squared-L2 top-k on the device in row blocks, ||q||^2 - 2 q.t + ||t||^2 like faiss's flat index: the
    k > 2 searches kernel 2 does not serve (k > 16, targets with fewer than k rows) and the reference the fused path is
    tested against."""
    k = min(k, t.shape[0])
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        tn = (t * t).sum(dim=1)
        ds, ids = [], []
        for r0 in range(0, q.shape[0], 4096):
            qb = q[r0:r0 + 4096]
            d2 = (qb * qb).sum(dim=1, keepdim=True) - 2.0 * (qb @ t.t()) + tn[None, :]
            d, i = torch.topk(d2, k, dim=1, largest=False, sorted=True)
            ds.append(d)
            ids.append(i)
        if not ds:
            return q.new_zeros((0, k)), torch.zeros((0, k), dtype=torch.int64, device=q.device)
        return torch.cat(ds), torch.cat(ids)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def knn_points(X_f, Y_f, K=1, metric="euclidean"):
    """(dists (N, K), idx (N, K) int64).  correspondence.py:26-60.

    cosine: rows are L2-normalised, neighbours come from kernel 2 and the distances 1 - cos are
    recomputed in fp32 by kernel 3, exactly the reference's order of operations (:47-58).
    euclidean: exact L2 neighbours through faiss_knn, distances = ||x - y||_2 (:55-56).
    3 <= K <= 16 (no call site in the reference) runs on kernel 2's row top-KP epilogue wherever there are at least K
    targets: euclidean through faiss_knn; cosine on the rows of the configured operand type (C % 8 == 0) with the fp32
    re-rank of mv_knn_rerank for the distances.  Other K > 2 take the exact blocked search of _exact_knn_blocks.
    """
    assert metric in ["cosine", "euclidean"]
    dev = _device()
    in_dev = X_f.device
    n, m = X_f.shape[0], Y_f.shape[0]
    fused = _fused_knn_applies(n, m, int(K)) and (metric == "euclidean" or X_f.shape[-1] % 8 == 0)
    if K > 2 and not fused:
        X, Y = _f32(X_f, dev), _f32(Y_f, dev)
        if metric == "cosine":
            X, Y = torch.nn.functional.normalize(X, dim=-1), torch.nn.functional.normalize(Y, dim=-1)
        _, idx = _exact_knn_blocks(X, Y, int(K))
        gathered = Y[idx]
        if metric == "euclidean":
            d = (gathered - X[:, None, :]).norm(p=2, dim=2)
        else:
            d = 1 - torch.nn.functional.cosine_similarity(gathered, X[:, None, :], dim=-1)
        return d.to(in_dev), idx.to(in_dev)
    if metric == "euclidean":
        _, idx = faiss_knn(X_f, Y_f, K)
        X = _f32(X_f, dev)
        Y = _f32(Y_f, dev)
        d = (Y[idx.to(dev)] - X[:, None, :]).norm(p=2, dim=2)
        return d.to(in_dev), idx
    if X_f.shape[0] == 0 or Y_f.shape[0] < K:
        raise ValueError(f"knn_points: {X_f.shape[0]} queries against {Y_f.shape[0]} targets for K={K}")
    (A16, A32), (B16, B32), mu = _rows_pair(X_f, Y_f, dev)
    if K > 2:
        A, B, Ck, dtype = _k2_operands(A16, A32, B16, B32, A32.shape[1])
        cand = _topk_candidates(A, B, n, m, Ck, dtype, int(K))
        d, idx = _rerank(A32, B32, cand, int(K), L.MV_METRIC_COSINE)
        return d.to(in_dev), idx.long().to(in_dev)
    r = match_rows(A16, A32, B16, B32, X_f.shape[0], Y_f.shape[0], 0, want_topk=False, center_B=mu)
    return r.dists[:, :K].to(in_dev), r.row_idx[:, :K].long().to(in_dev)


def get_correspondences_ratio_test(P1_F, P2_F, num_corres, metric="cosine", bidirectional=False, ratio_test=True):
    """(idx1, idx2, weight): the num_corres best matches by ratio weight.  correspondence.py:63-102.

    bidirectional=True follows the evident intent of the reference's (crashing, :96-98) branch: half the
    budget in each direction, concatenated.
    """
    assert metric in ["cosine", "euclidean"]
    if metric == "euclidean":
        return _ratio_test_euclidean(P1_F, P2_F, num_corres, bidirectional, ratio_test)
    dev = _device()
    in_dev = P1_F.device
    n, m = P1_F.shape[0], P2_F.shape[0]
    if n == 0 or m < 2:  # the reference's K=2 search has nothing to return (the dense helpers raise the same way)
        raise ValueError(f"get_correspondences_ratio_test: too few points to match ({n} vs {m})")
    (A16, A32), (B16, B32), mu = _rows_pair(P1_F, P2_F, dev)
    if not bidirectional:
        r = match_rows(A16, A32, B16, B32, n, m, num_corres, ratio_test, center_B=mu)
        k = r.k
        return (r.sel_src[:k].long().to(in_dev), r.sel_dst[:k].long().to(in_dev), r.sel_weight[:k].to(in_dev))
    r12 = match_rows(A16, A32, B16, B32, n, m, num_corres // 2, ratio_test, center_B=mu)
    (B16, B32), (A16, A32), mu = _rows_pair(P2_F, P1_F, dev)  # the reverse direction swaps the query / target roles
    r21 = match_rows(B16, B32, A16, A32, m, n, num_corres // 2, ratio_test, center_B=mu)
    idx1 = torch.cat((r12.sel_src[:r12.k], r21.sel_dst[:r21.k])).long()
    idx2 = torch.cat((r12.sel_dst[:r12.k], r21.sel_src[:r21.k])).long()
    w = torch.cat((r12.sel_weight[:r12.k], r21.sel_weight[:r21.k]))
    return idx1.to(in_dev), idx2.to(in_dev), w.to(in_dev)


def _ratio_test_euclidean(P1_F, P2_F, num_corres, bidirectional, ratio_test):
    """the metric="euclidean" branch (no call site in the reference; correspondence.py:70-102 followed literally):
    exact L2 2-NN (knn_points) -> ratio weights -> top-k through the library's selection kernel."""
    def one_way(X, Y, k):
        d, idx = knn_points(X, Y, 2, "euclidean")
        w = calculate_ratio_test(d) if ratio_test else d[:, 0]
        return get_topk_matches(w, idx[:, 0], k)

    if not bidirectional:
        return one_way(P1_F, P2_F, num_corres)
    a1, a2, aw = one_way(P1_F, P2_F, num_corres // 2)
    b2, b1, bw = one_way(P2_F, P1_F, num_corres // 2)
    return torch.cat((a1, b1)), torch.cat((a2, b2)), torch.cat((aw, bw))


def calculate_ratio_test(dists):
    """weight = 1 - d0 / d1 with both 1e-9 clamps.  correspondence.py:105-121 (runs inside kernel 3 on the
    matching path; this torch form serves callers that hold a (…, 2) distance tensor)."""
    d = dists.clamp(min=1e-9)
    return 1 - d[..., 0] / d[..., 1].clamp(min=1e-9)


def get_topk_matches(dists, idx, num_corres):
    """(idx_source, idx_target, dist) of the num_corres largest entries, sorted.  correspondence.py:125-129."""
    dev = _device()
    in_dev = dists.device
    w = _f32(dists, dev)
    n = w.shape[-1]
    pairs = torch.stack((idx.to(dev).to(torch.int32), torch.zeros(n, dtype=torch.int32, device=dev)), dim=1).contiguous()
    k = min(int(num_corres), n)
    src = _empty((max(k, 1),), torch.int32, dev)
    dst = _empty((max(k, 1),), torch.int32, dev)
    val = _empty((max(k, 1),), torch.float32, dev)
    L.call("mv_k3_topk_matches", L.ptr(w), L.ptr(pairs), None, n, int(num_corres), L.ptr(src), L.ptr(dst), L.ptr(val),
           None, _stream())
    return src[:k].long().to(in_dev), dst[:k].long().to(in_dev), val[:k].to(in_dev)


# ------------------------------------------------------------------------------------------------
# reference interface: geometry helpers
# ------------------------------------------------------------------------------------------------
def get_grid(H, W):
    """(3, H, W) pixel-centre grid (x + .5, y + .5, 1).  correspondence.py:132-144."""
    xs = torch.linspace(0.5, W - 0.5, W).view(1, W).expand(H, W)
    ys = torch.linspace(0.5, H - 0.5, H).view(H, 1).expand(H, W)
    return torch.stack((xs, ys, torch.ones(H, W)), dim=0).contiguous()


def grid_to_pointcloud(K_inv, depth, grid=None):
    """(H*W, 3) back-projection K^-1 (depth * grid).  correspondence.py:147-161."""
    _, H, W = depth.shape
    if grid is not None:  # caller-supplied grid: plain torch, same formula
        return (K_inv @ (depth * grid).reshape(3, H * W)).permute(1, 0)
    dev = _device()
    in_dev = depth.device
    d = _f32(depth, dev)
    Ki = L.host_floats(K_inv.detach().float().cpu().reshape(-1).tolist())
    out = _empty((H * W, 3), torch.float32, dev)
    L.call("mv_geom_backproject", L.ptr(d), H, W, Ki, L.ptr(out), _stream())
    return out.to(in_dev)


def sample_pointcloud_features(feats, K, pc, image_shape):
    """(n, C) bilinear samples of feats (C, h, w) at the projections of pc.  correspondence.py:164-176."""
    H, W = image_shape
    dev = _device()
    in_dev = feats.device
    src, C, h, w = _feature_map(feats, dev)
    p = _f32(pc, dev)
    n = p.shape[0]
    Kh = L.host_floats(K.detach().float().cpu().reshape(-1).tolist())
    xyz = _empty((max(n, 1), 3), torch.float32, dev)
    coords = _empty((max(n, 1), 2), torch.float32, dev)
    if n > 0:
        L.call("mv_geom_project_coords", L.ptr(p), None, None, n, Kh, int(H), int(W), h, w, L.ptr(xyz), L.ptr(coords),
               _stream())
    o32 = _sample(L.MV_SAMPLE_BILINEAR_ZEROS, src, C, h, w, coords, None, n, False, False, True)[1]
    return o32[:n].to(in_dev)


def argmax_2d(x, max_value=True):
    """(…, 2) int64 (col, row) of the arg-max (arg-min) over the last two dims.  correspondence.py:179-190."""
    dev = _device()
    in_dev = x.device
    h, w = x.shape[-2:]
    lead = x.shape[:-2]
    flat = _f32(x, dev).reshape(-1, h * w)
    rows = flat.shape[0]
    out = _empty((max(rows, 1),), torch.int32, dev)
    L.call("mv_argmax_rows", L.ptr(flat), rows, h * w, int(bool(max_value)), L.ptr(out), _stream())
    idx = out[:rows].long()
    xy = torch.stack((idx % w, idx // w), dim=-1).reshape(*lead, 2)
    return xy.to(in_dev)


def project_3dto2d(xyz, K_mat):
    """uv = (xyz K^T)[:, :2] / max(z', 1e-9).  correspondence.py:193-196 (same arithmetic inside mv_k3_score)."""
    uvd = xyz @ K_mat.transpose(-1, -2)
    return uvd[:, :2] / uvd[:, 2:3].clamp(min=1e-9)


def error_auc(errors, thresholds):
    """Area under the recall-vs-error curve up to each threshold, normalised.  correspondence.py:199-215."""
    errs = [0] + sorted(list(errors))
    recall = list(np.linspace(0, 1, len(errs)))
    trapz = getattr(np, "trapezoid", None) or np.trapz
    out = []
    for thr in thresholds:
        last = np.searchsorted(errs, thr)
        ys = recall[:last] + [recall[last - 1]]
        xs = errs[:last] + [thr]
        out.append(trapz(ys, xs) / thr)
    return out


def compute_binned_performance(y, x, x_bins):
    """mean of y over x in [x_bins[i], x_bins[i+1]).  correspondence.py:266-277."""
    return [y[(x >= lo) * (x < hi)].mean() for lo, hi in zip(x_bins[:-1], x_bins[1:])]


# ------------------------------------------------------------------------------------------------
# reference interface: the two dense helpers
# ------------------------------------------------------------------------------------------------
class _Side:
    """One image of a pair after kernel 1: compacted geometry + feature rows."""

    __slots__ = ("n", "n_dev", "xyz", "uv", "rows16", "rows32", "rows_lo", "valid_idx", "taps", "center",
                 "coords", "mode", "src", "fshape")  # the last four: what the low-rank proposal builds its operands from


def lowrank_applies(C, h, w, n_max, m_max, mode=L.MV_SAMPLE_BILINEAR_ZEROS):
    """whether the dense helpers run kernel 2 over the target's source pixels (h*w + 8 columns) instead of the channels."""
    cfg = _CFG["lowrank"]
    hwp = (h * w + 7) // 8 * 8
    if cfg == "0" or _CFG["dtype"] != "f16" or hwp > L.MV_LR_MAX_SOURCE_PIXELS or h * w < 2:
        return False
    if mode not in (L.MV_SAMPLE_BILINEAR_ZEROS, L.MV_SAMPLE_BICUBIC_CLAMP):
        return False
    if cfg == "1":
        return True
    # measured on B200: ScanNet-shaped (300 source pixels, C = 2048, 18231^2) 0.83 -> ~0.35 ms for kernel 2; NAVI-shaped (784
    # source pixels, C = 3072, 5024^2) would trade 113 us of kernel 2 for a 60 us product + a 45 us Gram launch + the builders
    return (hwp + 8) * 5 <= C and n_max * m_max >= (1 << 24)


def lowrank_exact_applies(C, h, w, n_max, m_max, mode=L.MV_SAMPLE_BILINEAR_ZEROS):
    """whether a dense helper runs WITHOUT kernel 1: low-rank proposal + kernel 3 on the exact Gram matrix of the source pixels."""
    return _CFG["lowrank_k3"] == "1" and C % 64 == 0 and _CFG["rows"] == "split" and lowrank_applies(C, h, w, n_max, m_max, mode)


def _lowrank_operands(s0, s1, n, m, n_dev, m_dev, exact=False):
    """fp16 operands of kernel 2 in the basis of the target image's source pixels (csrc/lr_gram.cu):
    unit source rows of both images -> their stacked cosine Gram matrix (kernel 2 with the similarity written out) ->
    query rows A' (n, P) and target rows B (m, P); returns (A', B, h*w padded + 8).
    exact=True: the Gram matrix of the RAW rows in fp32 from the CUDA cores instead (mv_lr_gram_exact); a fourth value is
    returned with what mv_k3_ratio_mutual_lr needs (G, its pitch, the points' inverse norms)."""
    C, h, w = s0.fshape
    dev = s0.src.device
    st = _stream()
    hw = h * w
    hwp = (hw + 7) // 8 * 8
    P = L.f16c_pitch(hwp)
    if exact:
        off1 = (hw + 31) // 32 * 32  # image 1's offset in the stacked Gram matrix: whole 32 x 32 tiles per image
        taps = 4 if s0.mode == L.MV_SAMPLE_BICUBIC_CLAMP else 2
        reach = (taps - 1) * (w + 1)  # largest index distance between two taps of one point
        G = _empty((2 * off1, 2 * off1), torch.float32, dev)
        snorm = _empty((2 * off1,), torch.float32, dev)
        rsnorm = _empty((2 * off1,), torch.float32, dev)
        L.call("mv_lr_gram_exact", L.ptr(s0.src), L.ptr(s1.src), C, hw, off1, reach, L.ptr(G), 2 * off1, L.ptr(snorm), L.ptr(rsnorm), st)
        A_op = _empty((max(n, 1), P), torch.float16, dev)
        B_op = _empty((max(m, 1), P), torch.float16, dev)
        inv0 = _empty((max(n, 1),), torch.float32, dev)
        inv1 = _empty((max(m, 1),), torch.float32, dev)
        L.call("mv_lr_build_target", s1.mode, L.ptr(s1.coords), L.ptr(m_dev), m, h, w, None, c_void_p(snorm.data_ptr() + off1 * 4),
               L.ptr(G), 2 * off1, off1, L.ptr(B_op), P, hwp, L.ptr(inv1), st)
        L.call("mv_lr_build_query", s0.mode, L.ptr(s0.coords), L.ptr(n_dev), n, h, w, None, c_void_p(rsnorm.data_ptr() + off1 * 4),
               L.ptr(G), 2 * off1, 0, off1, L.ptr(A_op), P, hwp, L.ptr(inv0), st)
        return A_op, B_op, hwp + 8, {"G": G, "ld": 2 * off1, "off_t": off1, "inv0": inv0, "inv1": inv1, "keep": (snorm, rsnorm)}
    U = _empty((2 * hwp, C), torch.float16, dev)
    if hwp > hw:  # pad rows: zero Gram rows / columns
        U[hw:hwp].zero_()
        U[hwp + hw:].zero_()
    snorm = _empty((2 * hwp,), torch.float32, dev)
    L.call("mv_lr_unit_rows", L.ptr(s0.src), C, hw, L.ptr(U), L.ptr(snorm), st)
    L.call("mv_lr_unit_rows", L.ptr(s1.src), C, hw, c_void_p(U.data_ptr() + hwp * C * 2), c_void_p(snorm.data_ptr() + hwp * 4), st)
    G = _empty((2 * hwp, 2 * hwp), torch.float32, dev)
    rv = _empty((2 * hwp, 2), torch.float32, dev)
    ri = _empty((2 * hwp, 2), torch.int32, dev)
    cb = _empty((2 * hwp,), torch.int64, dev)
    wsb = L.load().mv_k2_workspace_bytes(2 * hwp, 2 * hwp)
    ws = _empty((wsb,), torch.uint8, dev)
    L.call("mv_k2_affinity", L.ptr(U), C, L.ptr(U), C, 2 * hwp, 2 * hwp, C, None, None, L.MV_DTYPE_F16, _CFG["cluster"], L.ptr(G),
           2 * hwp, L.ptr(rv), L.ptr(ri), L.ptr(cb), L.ptr(ws), c_size_t(wsb), st)
    A_op = _empty((max(n, 1), P), torch.float16, dev)
    B_op = _empty((max(m, 1), P), torch.float16, dev)
    sn1 = c_void_p(snorm.data_ptr() + hwp * 4)
    L.call("mv_lr_build_target", s1.mode, L.ptr(s1.coords), L.ptr(m_dev), m, h, w, sn1, sn1, L.ptr(G),
           2 * hwp, hwp, L.ptr(B_op), P, hwp, None, st)
    L.call("mv_lr_build_query", s0.mode, L.ptr(s0.coords), L.ptr(n_dev), n, h, w, L.ptr(snorm), None, L.ptr(G), 2 * hwp, 0, hwp,
           L.ptr(A_op), P, hwp, None, st)
    return A_op, B_op, hwp + 8


def _match_lowrank_exact(s0, s1, n, m, num_corr, ratio_test=True, n_dev=None, m_dev=None, want_topk=True):
    """one directional match WITHOUT interpolated rows: kernel 2 on the low-rank operands, kernel 3's distances from the exact
    Gram matrix of the source pixels (mv_k3_ratio_mutual_lr), then the usual top-k.  Same MatchResult as match_rows."""
    dev = s0.src.device
    st = _stream()
    A_op, B_op, Ck, x = _lowrank_operands(s0, s1, n, m, n_dev, m_dev, exact=True)
    C, h, w = s0.fshape
    res = MatchResult()
    row_val = _empty((n, 2), torch.float32, dev)
    row_idx = _empty((n, 2), torch.int32, dev)
    col_best = _empty((m,), torch.int64, dev)
    ws_bytes = L.load().mv_k2_workspace_bytes(n, m)
    ws = _empty((ws_bytes,), torch.uint8, dev)
    prof = _PROFILE.get("k2_events")
    if prof is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    L.call("mv_k2_sim_top2_ld", L.ptr(A_op), A_op.shape[1], L.ptr(B_op), B_op.shape[1], n, m, Ck, L.ptr(n_dev), L.ptr(m_dev),
           L.MV_DTYPE_F16, _CFG["cluster"], L.ptr(row_val), L.ptr(row_idx), L.ptr(col_best), L.ptr(ws), c_size_t(ws_bytes), st)
    if prof is not None:
        ev1.record()
        prof.append((ev0, ev1, (n, m, Ck, n_dev, m_dev)))
    dists = _empty((n, 2), torch.float32, dev)
    weight = _empty((n,), torch.float32, dev)
    mutual = _empty((n,), torch.uint8, dev)
    L.call("mv_k3_ratio_mutual_lr", s0.mode, L.ptr(s0.coords), L.ptr(s1.coords), L.ptr(x["inv0"]), L.ptr(x["inv1"]), L.ptr(x["G"]),
           x["ld"], 0, x["off_t"], h, w, L.ptr(n_dev), n, L.ptr(row_idx), L.ptr(col_best), int(ratio_test), L.ptr(dists),
           L.ptr(weight), L.ptr(mutual), st)
    res.row_idx, res.dists, res.weight, res.mutual, res.col_best = row_idx, dists, weight, mutual, col_best
    if want_topk:
        k = min(int(num_corr), n)
        res.k = k
        res.sel_src = _empty((max(k, 1),), torch.int32, dev)
        res.sel_dst = _empty((max(k, 1),), torch.int32, dev)
        res.sel_weight = _empty((max(k, 1),), torch.float32, dev)
        res.k_dev = _empty((1,), torch.int32, dev)
        L.call("mv_k3_topk_matches", L.ptr(weight), L.ptr(row_idx), L.ptr(n_dev), n, k, L.ptr(res.sel_src),
               L.ptr(res.sel_dst), L.ptr(res.sel_weight), L.ptr(res.k_dev), st)
    return res


def _match_sides(s0, s1, n0, n1, num_corr, ratio_test=True, n_dev=None, m_dev=None):
    """s0 = query side, s1 = target side (prepared with the matching f16c roles, see _pair_maps)."""
    proposal = None
    if s0.rows16 is None and s0.rows32 is None:  # prepared without rows (want_rows=False): the exact low-rank route
        if not (s0.fshape == s1.fshape and s0.mode == s1.mode and s1.rows16 is None and s1.rows32 is None):
            raise ValueError("sides prepared without rows need equal feature shapes and sampling modes")
        return _match_lowrank_exact(s0, s1, n0, n1, num_corr, ratio_test, n_dev=n_dev, m_dev=m_dev)
    if (s0.src is not None and s1.src is not None and s0.fshape == s1.fshape and s0.mode == s1.mode and n0 > 0 and n1 > 0
            and s0.rows_lo is not None and lowrank_applies(*s0.fshape, n0, n1, s0.mode)):
        proposal = _lowrank_operands(s0, s1, n0, n1, n_dev, m_dev)
    return match_rows(s0.rows16, s0.rows32, s1.rows16, s1.rows32, n0, n1, num_corr, ratio_test, n_dev=n_dev, m_dev=m_dev,
                      A_lo=s0.rows_lo, B_lo=s1.rows_lo, center_B=s1.center, proposal=proposal)


def _pair_maps(feat_0, feat_1, dev, grid_pixels=0, mode=None):
    """channel-last fp32 maps of both images + the f16c centre of the target image (None for the other operand types):
    -> (fm0, fm1, kw0, kw1) where fm = (src, C, h, w) and kw are the role keywords of kernel 1 for each side.
    grid_pixels / mode: upper bound of the point count per image and the sampling mode -- where the exact low-rank route
    applies (lowrank_exact_applies) the sides are prepared WITHOUT rows (kw = want_rows False: no kernel 1, no centre)."""
    fm0, fm1 = _feature_map(feat_0, dev), _feature_map(feat_1, dev)
    if (mode is not None and fm0[1:] == fm1[1:]
            and lowrank_exact_applies(fm0[1], fm0[2], fm0[3], grid_pixels, grid_pixels, mode)):
        return fm0, fm1, {"want_rows": False}, {"want_rows": False}
    if _CFG["dtype"] == "bf16":
        return fm0, fm1, {}, {}
    mu = _center(fm1[0], fm1[0].shape[0], step=_center_step(fm1[0].shape[0]))
    return fm0, fm1, {"role": L.MV_ROLE_QUERY, "dotvec": mu, "pixdot": _rows_dot(fm0[0], mu)}, {"role": L.MV_ROLE_TARGET, "center": mu}


def _center_step(n_rows):
    """the centre only has to lie near the mean direction (the ranking is exact for every centre): ~256 pixels are plenty"""
    return max(1, n_rows // 256)


def _rows_dot(rows, vec):
    """(n,) fp32: rows[p] . vec (mv_rows_dot) -- the per-source-pixel dots kernel 1 blends into a query row's r."""
    out = _empty((rows.shape[0],), torch.float32, rows.device)
    L.call("mv_rows_dot", L.ptr(rows), rows.shape[1], rows.shape[0], L.ptr(vec), L.ptr(out), _stream())
    return out


def _stage_depth(depth_dev, Kinv):
    """back-projection + valid-pixel compaction of one image (launches only; the count stays on the device)."""
    H, W = depth_dev.shape[-2:]
    dev = depth_dev.device
    st = _stream()
    xyz_all = _empty((H * W, 3), torch.float32, dev)
    L.call("mv_geom_backproject", L.ptr(depth_dev), H, W, Kinv, L.ptr(xyz_all), st)
    valid_idx = _empty((H * W,), torch.int32, dev)
    n_dev = _empty((1,), torch.int32, dev)
    L.call("mv_compact_valid", c_void_p(xyz_all.data_ptr() + 8), 3, H * W, L.ptr(valid_idx), L.ptr(n_dev), st)
    return xyz_all, valid_idx, n_dev


def _finish_depth(f, d, K, staged, n, synced, want_taps=False, rows=None, role=L.MV_ROLE_QUERY, center=None, dotvec=None,
                  pixdot=None, want_rows=True):
    """projection to feature-map coordinates + kernel 1 for the n (live or upper-bound) points of one image.
    f: the (C, h, w) feature map in either layout (see _feature_map), or the tuple _feature_map returned for it."""
    xyz_all, valid_idx, n_dev = staged
    dev = d.device
    src, C, h, w = f if isinstance(f, tuple) else _feature_map(f, dev)
    H, W = d.shape[-2:]
    s = _Side()
    s.n_dev, s.valid_idx, s.n = n_dev, valid_idx, n
    nd = None if synced else n_dev
    s.xyz = _empty((max(n, 1), 3), torch.float32, dev)
    coords = _empty((max(n, 1), 2), torch.float32, dev)
    if n > 0:
        L.call("mv_geom_project_coords", L.ptr(xyz_all), L.ptr(valid_idx), L.ptr(nd), n, K, H, W, h, w, L.ptr(s.xyz),
               L.ptr(coords), _stream())
    s.taps = _empty((max(n, 1), 2), torch.int32, dev) if want_taps else None
    s.uv = None
    s.coords, s.mode, s.src, s.fshape = coords, L.MV_SAMPLE_BILINEAR_ZEROS, src, (C, h, w)
    s.center = None
    if not want_rows:  # the exact low-rank route: no interpolated rows at all
        s.rows16 = s.rows32 = s.rows_lo = None
        return s
    w16, w32, wlo = _row_format(rows)
    s.rows16, s.rows32, s.rows_lo = _sample(L.MV_SAMPLE_BILINEAR_ZEROS, src, C, h, w, coords, nd, n, True, w16, w32,
                                            s.taps, wlo, role=role, center=center, dotvec=dotvec, pixdot=pixdot)
    s.center = center
    return s


def prepare_depth_side(feat, depth, K, Kinv, dev, sync=True, want_taps=False, rows=None, **role_kw):
    """ScanNet-style preparation of one image.  correspondence.py:219-225, :147-176, :47-48.

    back-project depth -> keep z > 0 (row-major) -> project with K -> bilinear grid_sample coordinates
    (align_corners=False) -> kernel 1 (sample + L2 normalise).  sync=False keeps n on the device.
    """
    d = _f32(depth, dev)
    _check_C(feat[1] if isinstance(feat, tuple) else feat.shape[0])
    staged = _stage_depth(d, Kinv)
    n = int(staged[2].item()) if sync else d.shape[-2] * d.shape[-1]
    return _finish_depth(feat, d, K, staged, n, sync, want_taps, rows, **role_kw)


def _stage_xyz(g):
    """valid-pixel compaction of one (3, H, W) xyz grid (launch only)."""
    _, H, W = g.shape
    valid_idx = _empty((H * W,), torch.int32, g.device)
    n_dev = _empty((1,), torch.int32, g.device)
    L.call("mv_compact_valid", c_void_p(g.data_ptr() + 2 * H * W * 4), 1, H * W, L.ptr(valid_idx), L.ptr(n_dev), _stream())
    return valid_idx, n_dev


def _finish_xyz(f, g, staged, n, synced, want_taps=False, rows=None, role=L.MV_ROLE_QUERY, center=None, dotvec=None,
                pixdot=None, want_rows=True):
    valid_idx, n_dev = staged
    dev = g.device
    src, C, h, w = f if isinstance(f, tuple) else _feature_map(f, dev)
    _, H, W = g.shape
    s = _Side()
    s.n_dev, s.valid_idx, s.n = n_dev, valid_idx, n
    nd = None if synced else n_dev
    s.xyz = _empty((max(n, 1), 3), torch.float32, dev)
    s.uv = _empty((max(n, 1), 2), torch.float32, dev)
    coords = _empty((max(n, 1), 2), torch.float32, dev)
    if n > 0:
        L.call("mv_geom_grid_coords", L.ptr(g), L.ptr(valid_idx), L.ptr(nd), n, H, W, h, w, L.ptr(s.xyz), L.ptr(s.uv),
               L.ptr(coords), _stream())
    s.taps = _empty((max(n, 1), 2), torch.int32, dev) if want_taps else None
    s.coords, s.mode, s.src, s.fshape = coords, L.MV_SAMPLE_BICUBIC_CLAMP, src, (C, h, w)
    s.center = None
    if not want_rows:  # the exact low-rank route: no interpolated rows at all
        s.rows16 = s.rows32 = s.rows_lo = None
        return s
    w16, w32, wlo = _row_format(rows)
    s.center = center
    if (_CFG["k1_grid"] and _CFG["dtype"] == "f16" and w16 and wlo and not w32 and not want_taps and n > 0
            and L.load().mv_k1_grid_supported(C, h, w, H, W)):
        # f16c split rows of an integer-factor upsample: the tiled cluster kernel (a third of the L2 traffic)
        rank = _empty((H * W,), torch.int32, dev)
        L.call("mv_rank_of_valid", L.ptr(valid_idx), L.ptr(nd), n, L.ptr(rank), H * W, _stream())
        s.rows16 = _empty((n, L.f16c_pitch(C)), torch.float16, dev)
        s.rows_lo = _empty((n, C), torch.float16, dev)
        s.rows32 = None
        L.call("mv_k1_grid_f16c", L.ptr(src), C, h, w, H, W, L.ptr(rank), role, L.ptr(center), L.ptr(dotvec), L.ptr(s.rows16),
               s.rows16.shape[1], L.ptr(s.rows_lo), _stream())
        return s
    s.rows16, s.rows32, s.rows_lo = _sample(L.MV_SAMPLE_BICUBIC_CLAMP, src, C, h, w, coords, nd, n, True, w16, w32,
                                            s.taps, wlo, role=role, center=center, dotvec=dotvec, pixdot=pixdot)
    return s


def prepare_xyz_side(feat, xyz_grid, dev, sync=True, want_taps=False, rows=None, **role_kw):
    """NAVI-style preparation of one image.  correspondence.py:240-252, :47-48.

    bicubic upsample of feat to the xyz grid's size evaluated only at the pixels with xyz_grid[2] > 0
    (row-major), + their xyz and pixel-centre uv, + kernel 1's L2 normalisation.
    """
    g = _f32(xyz_grid, dev)
    _check_C(feat[1] if isinstance(feat, tuple) else feat.shape[0])
    staged = _stage_xyz(g)
    n = int(staged[1].item()) if sync else g.shape[-2] * g.shape[-1]
    return _finish_xyz(feat, g, staged, n, sync, want_taps, rows, **role_kw)


_SIDE_STREAMS = {}


def _on_side_stream(fn, dev):
    """run fn() (uploads + launches for the second image) on a side stream forked from the current stream, so
    its host -> device copies overlap the first image's kernels; the caller joins with _join_side()."""
    cur = torch.cuda.current_stream(dev)
    side = _SIDE_STREAMS.get(dev.index)
    if side is None:
        side = _SIDE_STREAMS[dev.index] = torch.cuda.Stream(device=dev)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        out = fn()
    return out, side


def _join_side(side, dev, *objs):
    cur = torch.cuda.current_stream(dev)
    cur.wait_stream(side)

    def rec(o):
        if torch.is_tensor(o):
            o.record_stream(cur)
        elif isinstance(o, (tuple, list)):
            for x in o:
                rec(x)
        elif hasattr(o, "__slots__"):
            for nme in o.__slots__:
                rec(getattr(o, nme, None))

    for o in objs:
        rec(o)


def _upload_feat(feat, dev):
    """feature map to the device, keeping a channel-last layout and a 16-bit dtype if it has them."""
    if _is_channel_last(feat) or feat.dtype in (torch.bfloat16, torch.float16):
        return feat.detach().to(device=dev, non_blocking=True)
    return _f32(feat, dev)


def _two_counts(a, b):
    """both live counts with a single device -> host read."""
    n0, n1 = torch.cat((a, b)).tolist()
    return int(n0), int(n1)


def _return_packed(parts, in_dev):
    """the helper's return tuple; for host callers one packed device -> host copy instead of one per tensor."""
    if in_dev.type == "cuda":
        return tuple(parts)
    widths = [p.shape[1] if p.dim() == 2 else 1 for p in parts]
    host = torch.cat([p.reshape(p.shape[0], -1) for p in parts], dim=1).to(in_dev)
    out, c = [], 0
    for p, wd in zip(parts, widths):
        blk = host[:, c:c + wd]
        out.append(blk.contiguous() if p.dim() == 2 else blk[:, 0].contiguous())
        c += wd
    return tuple(out)


def _host_mat(M):
    return L.host_floats(M.detach().float().cpu().reshape(-1).tolist())


def _graphed_helper(kind, feat_0, feat_1, grid_0, grid_1, num_corr, ratio_test, K=None):
    """Fast path of the two dense helpers: the whole pair (kernels 1-3 + the gathers of the return tuple) is one
    cached CUDA graph; a call is 4 copies into static buffers (uploads for host tensors), one replay and ONE
    packed read-back (results + the three live counts), i.e. a single host sync.  Results are returned on the
    device of the first feature argument, like the reference."""
    dev = _device()
    if tuple(feat_1.shape) != tuple(feat_0.shape) or tuple(grid_1.shape) != tuple(grid_0.shape):
        return None  # two differently sized images (the reference accepts them): the eager path handles any shapes
    layout = "hwc" if (_is_channel_last(feat_0) and _is_channel_last(feat_1)) else "chw"
    fdt = feat_0.dtype if (feat_0.dtype == feat_1.dtype and feat_0.dtype in _FEAT_DTYPES) else torch.float32
    on_host = feat_0.device.type == "cpu"
    # two graphs (upload of image 0 behind image 1's kernels): 1369 -> 1536 pairs/s NAVI-shaped from pinned sources; pageable
    # sources (staged by host threads, every CUDA call on this thread since round 2) gain 2 % (811 -> 829)
    split = on_host and bool(_CFG["helper_split"])
    # the intrinsics are NOT part of the key: they live in device memory and are refreshed per call (gm.load)
    key = (on_host, split, kind, tuple(feat_0.shape), tuple(grid_0.shape), int(num_corr), bool(ratio_test), _CFG["dtype"], _CFG["cluster"], _CFG["rows"], _CFG["k1_grid"], _CFG["lowrank"], _CFG["lowrank_k3"], fdt,
           dev.index, layout)
    gm = _HELPER_GRAPHS.get(key)
    if gm is None:
        import importlib

        ev = importlib.import_module(__package__ + ".evaluation")
        if len(_HELPER_GRAPHS) >= _HELPER_GRAPHS_MAX:
            _HELPER_GRAPHS.pop(next(iter(_HELPER_GRAPHS)))
        gm = ev.GraphedPairMatcher(kind, tuple(feat_0.shape), tuple(grid_0.shape), num_corr, K=K, device=dev,
                                   ratio_test=ratio_test, with_outputs=True, feat_layout=layout, feat_dtype=fdt,
                                   split=split).capture()
        _HELPER_GRAPHS[key] = gm
    if gm.split:  # host caller: image 1 uploads first and its side runs while image 0 uploads
        gm.load_and_replay_split(feat_0, feat_1, grid_0, grid_1, K=K)
    else:
        gm.load(feat_0, feat_1, grid_0, grid_1, two_streams=on_host, K=K)
        gm.graph.replay()
        L.LAUNCHES["count"] += gm.launches_per_replay
    if on_host:
        gm.host_packed.copy_(gm.packed, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        res = gm.host_packed.clone()  # the pinned buffer is overwritten by the next call
    else:  # device-resident caller (e.g. features straight from the backbone): results stay on its device
        res = gm.packed.clone()       # the static buffer is overwritten by the next replay
        if res.device != feat_0.device:
            res = res.to(feat_0.device)
    km = gm.k_max
    blocks = 11 if kind == "xyz" else 7
    n0, n1, k = (int(v) for v in res[blocks * km:blocks * km + 3].tolist())
    if n0 == 0 or n1 < 2:
        raise RuntimeError(f"too few valid points to match ({n0} vs {n1})")
    out = [res[0:3 * k].view(k, 3), res[3 * km:3 * km + 3 * k].view(k, 3), res[6 * km:6 * km + k]]
    if kind == "xyz":
        out += [res[7 * km:7 * km + 2 * k].view(k, 2), res[9 * km:9 * km + 2 * k].view(k, 2)]
    return tuple(out)


def estimate_correspondence_depth(feat_0, feat_1, depth_0, depth_1, K, num_corr=500):
    """(corr_xyz0 (k, 3), corr_xyz1 (k, 3), corr_dist (k,)).  correspondence.py:218-232."""
    dev = _device()
    in_dev = feat_0.device
    if _CFG["helper_graphs"]:
        out = _graphed_helper("depth", feat_0, feat_1, depth_0, depth_1, num_corr, True, K=K)
        if out is not None:
            return out
    Kc = K.detach().float().cpu()
    Kh, Kinv = _host_mat(Kc), _host_mat(Kc.inverse())
    _check_C(feat_0.shape[0])
    # the small depth maps go first (their compaction decides the point counts: one host read for both), then
    # image 1's feature upload rides a side stream and overlaps image 0's kernels
    d0, d1 = _f32(depth_0, dev), _f32(depth_1, dev)
    a0, a1 = _stage_depth(d0, Kinv), _stage_depth(d1, Kinv)
    n0, n1 = _two_counts(a0[2], a1[2])
    if n0 == 0 or n1 < 2:
        raise RuntimeError(f"too few valid points to match ({n0} vs {n1})")
    f0 = _upload_feat(feat_0, dev)
    f1, side = _on_side_stream(lambda: _upload_feat(feat_1, dev), dev)
    _join_side(side, dev, f1)  # the target's map is needed first: its centre goes into the query's rows (f16c)
    fm0, fm1, kw0, kw1 = _pair_maps(f0, f1, dev, max(n0, n1), L.MV_SAMPLE_BILINEAR_ZEROS)
    side.wait_stream(torch.cuda.current_stream(dev))
    s0 = _finish_depth(fm0, d0, Kh, a0, n0, True, **kw0)
    with torch.cuda.stream(side):
        s1 = _finish_depth(fm1, d1, Kh, a1, n1, True, **kw1)
    _join_side(side, dev, s1)
    r = _match_sides(s0, s1, n0, n1, num_corr)
    k = r.k
    return _return_packed([_gather(s0.xyz, r.sel_src, k), _gather(s1.xyz, r.sel_dst, k), r.sel_weight[:k]], in_dev)


def estimate_correspondence_xyz(feat_0, feat_1, xyz_grid_0, xyz_grid_1, num_corr=500, ratio_test=True):
    """(c_xyz0, c_xyz1, c_dist, c_uv0, c_uv1).  correspondence.py:235-263."""
    dev = _device()
    in_dev = feat_0.device
    if _CFG["helper_graphs"]:
        out = _graphed_helper("xyz", feat_0, feat_1, xyz_grid_0, xyz_grid_1, num_corr, ratio_test)
        if out is not None:
            return out
    _check_C(feat_0.shape[0])
    g0, g1 = _f32(xyz_grid_0, dev), _f32(xyz_grid_1, dev)
    a0, a1 = _stage_xyz(g0), _stage_xyz(g1)
    n0, n1 = _two_counts(a0[1], a1[1])
    if n0 == 0 or n1 < 2:
        raise RuntimeError(f"too few valid points to match ({n0} vs {n1})")
    f0 = _upload_feat(feat_0, dev)
    f1, side = _on_side_stream(lambda: _upload_feat(feat_1, dev), dev)
    _join_side(side, dev, f1)  # the target's map is needed first: its centre goes into the query's rows (f16c)
    fm0, fm1, kw0, kw1 = _pair_maps(f0, f1, dev, max(n0, n1), L.MV_SAMPLE_BICUBIC_CLAMP)
    side.wait_stream(torch.cuda.current_stream(dev))
    s0 = _finish_xyz(fm0, g0, a0, n0, True, **kw0)
    with torch.cuda.stream(side):
        s1 = _finish_xyz(fm1, g1, a1, n1, True, **kw1)
    _join_side(side, dev, s1)
    r = _match_sides(s0, s1, n0, n1, num_corr, ratio_test)
    k = r.k
    return _return_packed([_gather(s0.xyz, r.sel_src, k), _gather(s1.xyz, r.sel_dst, k), r.sel_weight[:k],
                           _gather(s0.uv, r.sel_src, k), _gather(s1.uv, r.sel_dst, k)], in_dev)
