"""TEST INFRASTRUCTURE ONLY -- CPU restatement (fp32 torch on the host) of the reference's matching path.

Each function names the reference lines it follows (paths relative to the reference project's root).  The k-NN
backend of the reference, faiss-gpu 1.8.0 GpuIndexFlatL2 (not in the tree; README.md:60), is restated
from its published behaviour: exact brute-force squared-L2 search, ascending, int64 labels.

Checked against (a) the reference's own module imported from a checkout of it (oracle/reference_loader.py; where present) and (b) the golden vectors
under tests/golden/ by tests/test_oracle.py.  Never imported by the product.
"""
import torch
import torch.nn.functional as F


# ---- k-NN ------------------------------------------------------------------------------------------
def exact_l2_knn(query, target, k):
    """faiss.GpuIndexFlatL2(res, d).add(target).search(query, k) -- evals/utils/correspondence.py:14-23."""
    q = query.contiguous().float()
    t = target.contiguous().float()
    d2 = (q * q).sum(1, keepdim=True) - 2.0 * (q @ t.t()) + (t * t).sum(1)[None, :]
    dist, idx = torch.topk(d2, k, dim=1, largest=False, sorted=True)
    return dist, idx


def knn_points(X_f, Y_f, K=1, metric="euclidean"):
    """evals/utils/correspondence.py:26-60: normalise (cosine), faiss indices, distances recomputed
    from the gathered rows (the faiss distances are discarded at :50)."""
    assert metric in ["cosine", "euclidean"]
    if metric == "cosine":
        X_f = F.normalize(X_f, dim=-1)
        Y_f = F.normalize(Y_f, dim=-1)
    _, nn_idx = exact_l2_knn(X_f, Y_f, K)
    gathered = Y_f[nn_idx]                                   # (N, K, C)   :53
    if metric == "euclidean":
        dists = (gathered - X_f[:, None, :]).norm(p=2, dim=2)  # :55-56 (the reference's dim=3 is a bug there)
    else:
        dists = 1 - F.cosine_similarity(gathered, X_f[:, None, :], dim=-1)  # :58
    return dists, nn_idx


def ratio_weights(dists):
    """calculate_ratio_test, evals/utils/correspondence.py:105-121."""
    d = dists.clamp(min=1e-9)
    return 1 - d[..., 0] / d[..., 1].clamp(min=1e-9)


def topk_matches(weights, idx, num_corres):
    """get_topk_matches, evals/utils/correspondence.py:125-129."""
    k = min(num_corres, weights.shape[-1])
    w, src = torch.topk(weights, k=k, dim=-1)
    return src, idx[src], w


def correspondences_ratio_test(P1_F, P2_F, num_corres, ratio_test=True, return_all=False):
    """get_correspondences_ratio_test with bidirectional=False, evals/utils/correspondence.py:63-102."""
    dists, idx = knn_points(P1_F, P2_F, 2, "cosine")
    w = ratio_weights(dists) if ratio_test else dists[:, 0]
    out = topk_matches(w, idx[:, 0], num_corres)
    if return_all:
        return out + (dists, idx, w)
    return out


def similarity_top2_and_mutual(X_f, Y_f):
    """What kernel 2 adds on top of the reference: fp32 cosine similarities of the normalised rows, the
    two best columns per row (ties to the lower column), the best row per column, the mutual flag and
    the top-2 similarity gap used by the north-star tolerance."""
    Xn = F.normalize(X_f.float(), dim=-1)
    Yn = F.normalize(Y_f.float(), dim=-1)
    S = Xn @ Yn.t()
    val, idx = torch.topk(S, min(2, S.shape[1]), dim=1)
    col_val, col_idx = S.max(dim=0)
    mutual = col_idx[idx[:, 0]] == torch.arange(S.shape[0])
    gap = val[:, 0] - val[:, 1] if S.shape[1] > 1 else torch.full((S.shape[0],), float("inf"))
    col_sorted = torch.topk(S, min(2, S.shape[0]), dim=0).values
    col_gap = col_sorted[0] - col_sorted[1] if S.shape[0] > 1 else torch.full((S.shape[1],), float("inf"))
    return {"S": S, "row_val": val, "row_idx": idx, "col_val": col_val, "col_idx": col_idx, "mutual": mutual,
            "row_gap": gap, "col_gap": col_gap}


# ---- geometry + sampling ---------------------------------------------------------------------------
def pixel_grid(H, W):
    """get_grid, evals/utils/correspondence.py:132-144."""
    xs = torch.linspace(0.5, W - 0.5, W).view(1, W).repeat(H, 1)
    ys = torch.linspace(0.5, H - 0.5, H).view(H, 1).repeat(1, W)
    return torch.stack((xs, ys, torch.ones_like(xs)), dim=0)


def backproject(K_inv, depth):
    """grid_to_pointcloud, evals/utils/correspondence.py:147-161."""
    _, H, W = depth.shape
    pts = (depth * pixel_grid(H, W)).view(3, H * W)
    return (K_inv @ pts).permute(1, 0)


def depth_side_coords(K, pc, image_shape, feat_hw):
    """The projection + NDC step of sample_pointcloud_features (:164-170) followed by grid_sample's own
    align_corners=False un-normalisation on the CPU (ATen GridSamplerKernel.cpp: (g + 1) * (size / 2) - 0.5).
    Returns the continuous source coordinates (ix, iy) whose floor is the tap origin."""
    H, W = image_shape
    h, w = feat_hw
    uvd = pc @ K.transpose(-1, -2)
    uv = uvd[:, :2] / uvd[:, 2:3].clamp(min=1e-9)
    gx = (2 * uv[:, 0] / W) - 1
    gy = (2 * uv[:, 1] / H) - 1
    return torch.stack(((gx + 1) * (w / 2) - 0.5, (gy + 1) * (h / 2) - 0.5), dim=1)


def sample_pointcloud_features(feats, K, pc, image_shape):
    """evals/utils/correspondence.py:164-176."""
    H, W = image_shape
    uvd = pc @ K.transpose(-1, -2)
    uv = uvd[:, :2] / uvd[:, 2:3].clamp(min=1e-9)
    uv = torch.stack(((2 * uv[:, 0] / W) - 1, (2 * uv[:, 1] / H) - 1), dim=1)
    out = F.grid_sample(feats[None], uv[None, None], align_corners=False)
    return out[:, :, 0].transpose(1, 2)[0]


def depth_side(feat, depth, K):
    """One image of estimate_correspondence_depth (:219-225): (xyz (n, 3), features (n, C), valid index)."""
    xyz_all = backproject(K.inverse(), depth)
    keep = xyz_all[:, 2] > 0
    xyz = xyz_all[keep]
    return xyz, sample_pointcloud_features(feat, K.clone(), xyz, depth.shape[-2:]), keep.nonzero().squeeze(1)


def xyz_side(feat, xyz_grid):
    """One image of estimate_correspondence_xyz (:239-252): bicubic upsample, keep xyz_grid[2] > 0."""
    _, h, w = xyz_grid.shape
    up = F.interpolate(feat[None], size=(h, w), mode="bicubic")[0]
    keep = xyz_grid[2] > 0
    uvd = pixel_grid(h, w).to(xyz_grid)
    return (xyz_grid.permute(1, 2, 0)[keep], up.permute(1, 2, 0)[keep], uvd.permute(1, 2, 0)[keep][:, :2],
            keep.flatten().nonzero().squeeze(1))


def estimate_correspondence_depth(feat_0, feat_1, depth_0, depth_1, K, num_corr=500):
    """evals/utils/correspondence.py:218-232."""
    xyz_0, f_0, _ = depth_side(feat_0, depth_0, K)
    xyz_1, f_1, _ = depth_side(feat_1, depth_1, K)
    i0, i1, w = correspondences_ratio_test(f_0, f_1, num_corr)
    return xyz_0[i0], xyz_1[i1], w


def estimate_correspondence_xyz(feat_0, feat_1, xyz_grid_0, xyz_grid_1, num_corr=500, ratio_test=True):
    """evals/utils/correspondence.py:235-263."""
    xyz_0, f_0, uv_0, _ = xyz_side(feat_0, xyz_grid_0)
    xyz_1, f_1, uv_1, _ = xyz_side(feat_1, xyz_grid_1)
    i0, i1, w = correspondences_ratio_test(f_0, f_1, num_corr, ratio_test)
    return xyz_0[i0], xyz_1[i1], w, uv_0[i0], uv_1[i1]


def argmax_2d(x, max_value=True):
    """evals/utils/correspondence.py:179-190."""
    w = x.shape[-1]
    flat = torch.flatten(x, start_dim=-2)
    idx = flat.argmax(dim=-1) if max_value else flat.argmin(dim=-1)
    return torch.stack((idx % w, idx // w), dim=-1)


# ---- errors / recall --------------------------------------------------------------------------------
def transform_points_Rt(points, Rt):
    """evals/utils/transformations.py:27-36 (inverse=False)."""
    return points @ Rt[..., :3, :3].transpose(-2, -1) + Rt[..., None, :3, 3]


def project_3dto2d(xyz, K_mat):
    """evals/utils/correspondence.py:193-196."""
    uvd = xyz @ K_mat.transpose(-1, -2)
    return uvd[:, :2] / uvd[:, 2:3].clamp(min=1e-9)


def pair_errors(c_xyz0, c_xyz1, Rt, K_mat):
    """3-D and 2-D errors of one pair: evaluate_navi_correspondence.py:186-191,
    render_scannet_correspondence.py:211-217."""
    x0in1 = transform_points_Rt(c_xyz0, Rt.float())
    e3 = (x0in1 - c_xyz1).norm(p=2, dim=1)
    e2 = (project_3dto2d(x0in1, K_mat) - project_3dto2d(c_xyz1, K_mat)).norm(p=2, dim=1)
    return e3, e2


def recall(errors, thresholds):
    """100 * (err < th).float().mean(): evaluate_navi_correspondence.py:200-212."""
    return [100.0 * (errors < t).float().mean().item() for t in thresholds]


# ---- SPair -------------------------------------------------------------------------------------------
def spair_compute_errors(feats, kps_i, kps_j, thresh_scale, image_size, return_pred=False):
    """evaluate_spair_correspondence.py:59-103 with the backbone output `feats` (2, C, h, w) as input."""
    feats = F.normalize(feats.float(), p=2, dim=1)                      # :59
    fi, fj = feats[0], feats[1]
    kps_i = kps_i.clone().float()
    kps_j = kps_j.clone().float()
    kps_i[:, :2] = kps_i[:, :2] / image_size                            # :71-72
    kps_j[:, :2] = kps_j[:, :2] / image_size
    ndc = (kps_i[:, :2] * 2 - 1)[None, None]                            # :75
    kp_F = F.grid_sample(fi[None], ndc, mode="bilinear", align_corners=True)[0, :, 0].t()  # :76-79
    heat = torch.einsum("kf,fhw->khw", kp_F, fj)                        # :82
    pred = argmax_2d(heat).float() / feats.shape[-1]                    # :83
    errors = (pred[:, None, :] - kps_j[None, :, :2]).norm(p=2, dim=-1) / thresh_scale  # :86-87
    valid = (kps_i[:, None, 2] * kps_j[None, :, 2]) == 1                # :90
    in_both = valid.diagonal()
    errors[valid.logical_not()] = 1e3                                   # :94
    error_same = errors.diagonal()[in_both]                             # :96
    error_nn, index_nn = errors[in_both].min(dim=1)                     # :97
    index_same = in_both.nonzero().squeeze(1)                           # :98
    if return_pred:
        return error_same, error_nn, index_same, index_nn, heat
    return error_same, error_nn, index_same, index_nn


# ---- the two reference entry points without a caller ---------------------------------------------------
def correspondences_ratio_test_bidirectional(P1_F, P2_F, num_corres, ratio_test=True):
    """get_correspondences_ratio_test with bidirectional=True, evals/utils/correspondence.py:79-98, with the
    concatenations along dim 0 (the reference's `dim=1` on these 1-D tensors raises; dim 0 is what the surrounding code
    -- half the budget per direction, then one list of matches -- evidently means)."""
    d1, i1 = knn_points(P1_F, P2_F, 2, "cosine")
    d2, i2 = knn_points(P2_F, P1_F, 2, "cosine")
    w1 = ratio_weights(d1) if ratio_test else d1[:, 0]
    w2 = ratio_weights(d2) if ratio_test else d2[:, 0]
    m12_idx1, m12_idx2, m12_dist = topk_matches(w1, i1[:, 0], num_corres // 2)   # :89-91
    m21_idx2, m21_idx1, m21_dist = topk_matches(w2, i2[:, 0], num_corres // 2)   # :92-94
    return torch.cat((m12_idx1, m21_idx1)), torch.cat((m12_idx2, m21_idx2)), torch.cat((m12_dist, m21_dist))


def error_auc(errors, thresholds):
    """evals/utils/correspondence.py:199-215 (numpy; no caller in the reference)."""
    import numpy as np

    errors = [0] + sorted(list(errors))
    recall = list(np.linspace(0, 1, len(errors)))
    trapz = getattr(np, "trapezoid", None) or np.trapz
    aucs = []
    for thr in thresholds:
        last_index = np.searchsorted(errors, thr)
        y = recall[:last_index] + [recall[last_index - 1]]
        x = errors[:last_index] + [thr]
        aucs.append(trapz(y, x) / thr)
    return aucs


# ---- a caller, restated: the NAVI evaluation loop -------------------------------------------------------
def navi_error_block(corr, tr, feats_0, feats_1, xyz_grid_0, xyz_grid_1, Rt_gt, intrinsics, num_corr, scale_factor=0.25):
    """evaluate_navi_correspondence.py:174-221 with the functions taken from the modules `corr` (an
    evals.utils.correspondence) and `tr` (an evals.utils.transformations): the per-pair helper call, the 3-D / 2-D
    errors, the six recalls and the angle-binned recall@2cm.  Pinned against the reference's own text by
    tests/test_oracle.py (oracle/reference_loader.navi_error_block_reference executes those lines)."""
    import math

    err_3d, err_2d = [], []
    for i in range(len(feats_0)):                                                     # :177
        c_xyz0, c_xyz1, c_dist, c_uv0, c_uv1 = corr.estimate_correspondence_xyz(      # :178-180
            feats_0[i], feats_1[i], xyz_grid_0[i], xyz_grid_1[i], num_corr)
        c_uv0, c_uv1 = c_uv0 / scale_factor, c_uv1 / scale_factor                     # :182-183
        c_xyz0in1 = tr.transform_points_Rt(c_xyz0, Rt_gt[i].float())                  # :185
        c_err3d = (c_xyz0in1 - c_xyz1).norm(p=2, dim=1)                               # :186
        uv1 = corr.project_3dto2d(c_xyz1, intrinsics[i])                              # :188
        uv0 = corr.project_3dto2d(c_xyz0in1, intrinsics[i])                           # :189
        c_err2d = (uv0 - uv1).norm(p=2, dim=1)                                        # :190
        err_3d.append(c_err3d.detach().cpu())
        err_2d.append(c_err2d.detach().cpu())
    err_3d = torch.stack(err_3d, dim=0).float()                                       # :195-196
    err_2d = torch.stack(err_2d, dim=0).float()
    rec3 = [100 * (err_3d < th).float().mean() for th in (0.01, 0.02, 0.05)]          # :199-204
    rec2 = [100 * (err_2d < th).float().mean() for th in (5, 25, 50)]                 # :206-211
    rel_ang = tr.so3_rotation_angle(Rt_gt[:, :3, :3]) * 180.0 / math.pi              # :214-215
    rec_2cm = (err_3d < 0.02).float().mean(dim=1)                                     # :218
    bin_rec = corr.compute_binned_performance(rec_2cm, rel_ang, [0, 30, 60, 90, 120]) # :219
    return {"err_3d": err_3d, "err_2d": err_2d, "recall_3d": torch.stack(rec3), "recall_2d": torch.stack(rec2),
            "bin_rec": torch.stack([torch.as_tensor(b) for b in bin_rec])}


def compute_binned_performance(y, x, x_bins):
    """evals/utils/correspondence.py:266-277."""
    return [y[(x >= x_bins[i]) * (x < x_bins[i + 1])].mean() for i in range(len(x_bins) - 1)]


def so3_rotation_angle(R, eps=1e-4):
    """evals/utils/transformations.py:47-63: rotation angle (radians) of a batch of 3x3 rotations from the trace."""
    tr = R[:, 0, 0] + R[:, 1, 1] + R[:, 2, 2]
    if ((tr < -1.0 - eps) + (tr > 3.0 + eps)).any():
        raise ValueError("A matrix has trace outside valid range [-1-eps,3+eps].")
    return torch.acos(((tr - 1.0) * 0.5).clamp(min=-1, max=1))


# ---- the adjacent similarity consumers (SURVEY 8f.4) ---------------------------------------------------
def maskcut_affinity(feats, tau=None, eps=1e-5):
    """evals/models/maskcut_processor.py:77-78 (normalised affinity of the columns of feats (C, N)) and, for a given
    tau, :103-106 (A = A > tau; zeros -> eps; d_i = row sums).  The k-means choice of tau (:80-96) is not restated."""
    f = F.normalize(feats.float(), p=2, dim=0)
    A = f.transpose(0, 1) @ f
    if tau is None:
        return A
    B = (A > tau).double()
    B = torch.where(B == 0, torch.full_like(B, eps), B)
    return A, B, B.sum(dim=1)


def twoafc(features_ref, features_left, features_right):
    """evaluate_model_percepture.py:46-48, :118-122."""
    sl = F.cosine_similarity(features_ref, features_left, dim=-1)
    sr = F.cosine_similarity(features_ref, features_right, dim=-1)
    return sl, sr, torch.where(sl > sr, 0, 1)
