"""SPair-71k keypoint transfer on the B200 path: the matching lines that the reference inlines in
``evaluate_spair_correspondence.py:compute_errors`` (:59-103), taking the backbone's features instead
of the model so that the frozen forward stays in PyTorch.

    feats (2, C, h, w)  ->  per-pixel L2 normalise (:59)  ->  bilinear keypoint gather, align_corners=True
    (:71-79)  ->  K x (h*w) similarity + arg-max (:82-83, kernel 2)  ->  error matrix / thresh_scale,
    validity, error_same / error_nn (:86-98, kernel 3)  ->  PCK hit counts (:121)
"""
from ctypes import c_float, c_size_t

import torch

from . import _lib as L
from . import correspondence as C_

__all__ = ["compute_errors_from_features", "compute_errors_batch", "evaluate_pairs", "evaluate_batches", "pck_recall"]


def compute_errors_from_features(feats, kps_i, kps_j, thresh_scale, image_size, pck_thresh=0.10, hits=None,
                                 return_heatmap_argmax=False, confusion=None):
    """(error_same, error_nn, index_same, index_nn), as compute_errors (evaluate_spair_correspondence.py:45-103).

    feats: (2, C, h, w) backbone output for (image_i, image_j); kps_*: (K, 3) = (x, y, valid) in image
    pixels; image_size: side of the (square) input image.  hits: optional int64[2] device tensor that
    accumulates (#keypoints in both images, #of those with error_same < pck_thresh).  confusion: optional
    (D, D) int64 device tensor, D >= K, accumulating confusion[src, tgt] += 1 over (index_same, index_nn)
    (evaluate_dataset, evaluate_spair_correspondence.py:115-118).
    """
    dev = C_._device()
    in_dev = kps_i.device
    st = C_._stream()
    f = C_._f32(feats, dev)
    _, C, h, w = f.shape
    C_._check_C(C)
    ki = C_._f32(kps_i, dev)
    kj = C_._f32(kps_j, dev)
    K = ki.shape[0]
    if K > 64:
        raise ValueError("at most 64 keypoint slots")
    want16 = C_._CFG["dtype"] != "tf32"
    src_i = C_._hwc(f[0], prenorm=True)
    rows_j32 = C_._hwc(f[1], prenorm=True)  # (h*w, C): the heat-map columns, pixel p = y*w + x
    coords = torch.empty((K, 2), dtype=torch.float32, device=dev)
    L.call("mv_geom_keypoint_coords", L.ptr(ki), ki.shape[1], K, c_float(float(image_size)), h, w, L.ptr(coords), st)
    # f16c operands: image j's pixels are the targets (stored relative to their centre), the key-point rows the queries
    mu = C_._center(rows_j32, h * w) if C_._CFG["dtype"] != "bf16" else None
    a16, a32, _ = C_._sample(L.MV_SAMPLE_BILINEAR_ZEROS, src_i, C, h, w, coords, None, K, False, want16, True,
                             role=L.MV_ROLE_QUERY, dotvec=mu)
    b16 = None
    if want16 or mu is not None:  # the kernel-2 operand rows of image j (bf16 / f16c / tf32c)
        b16 = C_._sample(L.MV_SAMPLE_ROWS, rows_j32, C, 0, 0, None, None, h * w, False, want16, not want16,
                         role=L.MV_ROLE_TARGET, center=mu)[0]
    r = C_.match_rows(a16, a32, b16, rows_j32, K, h * w, 0, want_topk=False, center_B=mu)
    pred = r.row_idx[:, 0].contiguous()
    err_same = torch.empty((K,), dtype=torch.float32, device=dev)
    err_nn = torch.empty((K,), dtype=torch.float32, device=dev)
    idx_nn = torch.empty((K,), dtype=torch.int32, device=dev)
    L.call("mv_k3_spair_errors", L.ptr(pred), K, w, L.ptr(ki), L.ptr(kj), ki.shape[1], c_float(float(image_size)),
           c_float(float(thresh_scale)), c_float(float(pck_thresh)), None, L.ptr(err_same), L.ptr(err_nn),
           L.ptr(idx_nn), L.ptr(hits), L.ptr(confusion), 0 if confusion is None else confusion.shape[1], st)
    in_both = err_same >= 0
    out = (err_same[in_both].to(in_dev), err_nn[in_both].to(in_dev), in_both.nonzero().squeeze(1).to(in_dev),
           idx_nn[in_both].long().to(in_dev))
    if return_heatmap_argmax:
        return out + (pred.long().to(in_dev),)
    return out


def compute_errors_batch(feats, kps_i, kps_j, thresh_scale, image_size, pck_thresh=0.10, hits=None, confusion=None):
    """compute_errors (evaluate_spair_correspondence.py:45-103) for a whole batch of pairs in ONE launch.

    feats: (B, 2, C, h, w) backbone output of the B pairs (image_i, image_j); kps_i / kps_j: (B, K, 3);
    thresh_scale: (B,) tensor or sequence.  Returns device tensors (error_same, error_nn, index_nn, pred), each
    (B, K): entries of key points that are not in both images are -1 (the reference drops them, :96-98);
    pred is the flat arg-max pixel of each heat map (:83).  hits / confusion accumulate like
    compute_errors_from_features.  Nothing syncs.

    A bf16 or fp16 feats (an autocast backbone's output, on the host or the device) is uploaded and made contiguous as
    it is, and the kernel reads the 16-bit map (mv_spair_match_batch_typed): half the bytes, widened exactly on the chip,
    and the same results, bit for bit, as for feats.float().  Any other dtype is converted to fp32 first.  The key
    points and the arithmetic are fp32 throughout.
    """
    dev = C_._device()
    st = C_._stream()
    f16 = feats.dtype in (torch.bfloat16, torch.float16)
    f = feats.detach().to(device=dev, non_blocking=True).contiguous() if f16 else C_._f32(feats, dev)
    B, two, C, h, w = f.shape
    if two != 2:
        raise ValueError("feats must be (B, 2, C, h, w)")
    ki = C_._f32(kps_i, dev)
    kj = C_._f32(kps_j, dev)
    K = ki.shape[1]
    if K > 64:
        raise ValueError("at most 64 keypoint slots")
    if ki.shape != kj.shape or ki.shape[0] != B or ki.shape[2] < 3:
        raise ValueError("kps_i / kps_j must both be (B, K, >= 3)")
    ts = C_._f32(torch.as_tensor(thresh_scale, dtype=torch.float32).reshape(-1), dev)
    if ts.numel() != B:
        raise ValueError("thresh_scale needs one entry per pair")
    pred = torch.empty((B, K), dtype=torch.int32, device=dev)
    err_same = torch.empty((B, K), dtype=torch.float32, device=dev)
    err_nn = torch.empty((B, K), dtype=torch.float32, device=dev)
    idx_nn = torch.empty((B, K), dtype=torch.int32, device=dev)
    rest = (B, C, h, w, L.ptr(ki), L.ptr(kj), K, ki.shape[2], L.ptr(ts), c_float(float(image_size)),
            c_float(float(pck_thresh)), L.ptr(pred), L.ptr(err_same), L.ptr(err_nn), L.ptr(idx_nn), L.ptr(hits),
            L.ptr(confusion), 0 if confusion is None else confusion.shape[1], st)
    if f16:
        L.call("mv_spair_match_batch_typed", L.ptr(f), C_._FEAT_DTYPES[f.dtype], *rest)
    else:
        L.call("mv_spair_match_batch", L.ptr(f), *rest)
    return err_same, err_nn, idx_nn, pred


def set_heatmap_precision(mode):
    """Precision of compute_errors_batch's heat map (the einsum of evaluate_spair_correspondence.py:82) on the tensor cores:
    "3xtf32" (default; ~21 mantissa bits, arg-max equal to the fp32 reference's wherever its top-2 gap exceeds 1e-5) or
    "tf32" (one MMA per tile: operands rounded to 10 mantissa bits, fp32 accumulation -- equal wherever the gap exceeds
    1e-3, the tolerance of the matching path's tf32 operand type).  Returns the previous mode."""
    terms = {"3xtf32": 3, "tf32": 1}[mode]
    prev = L.load().mv_spair_set_heatmap_terms(terms)
    return "tf32" if prev == 1 else "3xtf32"


def evaluate_batches(batches, pck_thresh=0.10, kp_max=30):
    """(recall, confusion) over an iterable of dicts with keys feats (B, 2, C, h, w), kps_i, kps_j (B, K, 3),
    thresh_scale (B), image_size: evaluate_dataset (evaluate_spair_correspondence.py:106-123) with one launch per
    batch of pairs and integer counts; a single device -> host read at the end."""
    dev = C_._device()
    hits = torch.zeros(2, dtype=torch.int64, device=dev)
    conf = torch.zeros((kp_max, kp_max), dtype=torch.int64, device=dev)
    for b in batches:
        compute_errors_batch(b["feats"], b["kps_i"], b["kps_j"], b["thresh_scale"], b["image_size"],
                             pck_thresh=pck_thresh, hits=hits, confusion=conf)
    return pck_recall(hits), conf.cpu()


def evaluate_pairs(pairs, pck_thresh=0.10, kp_max=None):
    """(recall, confusion) over an iterable of dicts with keys feats, kps_i, kps_j, thresh_scale, image_size:
    evaluate_dataset (evaluate_spair_correspondence.py:106-123) on integer counts, nothing leaves the device
    until the end."""
    dev = C_._device()
    pairs = list(pairs)
    D = kp_max or max(int(p["kps_i"].shape[0]) for p in pairs)
    hits = torch.zeros(2, dtype=torch.int64, device=dev)
    conf = torch.zeros((D, D), dtype=torch.int64, device=dev)
    for p in pairs:
        compute_errors_from_features(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"],
                                     pck_thresh=pck_thresh, hits=hits, confusion=conf)
    return pck_recall(hits), conf.cpu()


def pck_recall(hits):
    """100 * hits[1] / hits[0]  (evaluate_spair_correspondence.py:121 on the integer counts)."""
    h = hits.tolist()
    return 100.0 * h[1] / max(h[0], 1)
