"""Pin oracle/restated.py: against the golden vectors produced by the reference's own module
(tests/golden, made by oracle/make_golden.py) and, where a checkout of the reference is present (oracle/_ref/ or
$MV_REFERENCE_ROOT, oracle/reference_loader.py), against that module directly on fresh inputs."""
import numpy as np
import pytest
import torch

from oracle import reference_loader, restated

SCANNET_SMALL = dict(C=64, h=6, w=8, H=24, W=32)
NAVI_SMALL = dict(C=64, h=8, w=8, H=32, W=32, radius=12.0)
SPAIR_SMALL = dict(C=64, h=14, w=14, K=20, image_size=224)
# error_auc([0.3, 4.0, 1.2, 9.5, 0.05, 2.2, 7.7, 3.1], [1, 5, 10]) of the reference (evals/utils/correspondence.py:199-215)
ERROR_AUC_GOLDEN = [0.22499999999999998, 0.5287499999999999, 0.70875]


def t(a):
    return torch.from_numpy(np.asarray(a))


@pytest.mark.parametrize("tag,coherent", [("coh", True), ("rnd", False)])
def test_scannet_golden(golden, syn, tag, coherent):
    g = golden(f"scannet_small_{tag}")
    p = syn.scannet_pair(7, coherent=coherent, **SCANNET_SMALL)
    assert np.isclose(p["feat_0"].double().sum().item(), float(g["feat_checksum"]), rtol=0, atol=1e-6)
    x0, x1, w = restated.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 100)
    torch.testing.assert_close(w, t(g["corr_dist"]), rtol=0, atol=2e-6)
    torch.testing.assert_close(x0, t(g["corr_xyz0"]), rtol=0, atol=0)
    torch.testing.assert_close(x1, t(g["corr_xyz1"]), rtol=0, atol=0)
    pc = restated.backproject(p["K"].inverse(), p["depth_0"])
    torch.testing.assert_close(pc, t(g["pointcloud"]), rtol=0, atol=0)
    xyz, f, _ = restated.depth_side(p["feat_0"], p["depth_0"], p["K"])
    torch.testing.assert_close(f, t(g["sampled"]), rtol=0, atol=1e-6)
    e3, _ = restated.pair_errors(x0, x1, p["Rt"], p["K"])
    torch.testing.assert_close(e3, t(g["err3d"]), rtol=0, atol=1e-6)


@pytest.mark.parametrize("tag,coherent", [("coh", True), ("rnd", False)])
def test_navi_golden(golden, syn, tag, coherent):
    g = golden(f"navi_small_{tag}")
    p = syn.navi_pair(7, coherent=coherent, **NAVI_SMALL)
    out = restated.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 100)
    for a, key in zip(out, ["c_xyz0", "c_xyz1", "c_dist", "c_uv0", "c_uv1"]):
        torch.testing.assert_close(a, t(g[key]), rtol=0, atol=2e-6 if key == "c_dist" else 0)
    nr = restated.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 100, ratio_test=False)
    torch.testing.assert_close(nr[2], t(g["nr_dist"]), rtol=0, atol=2e-6)


def test_rows_golden(golden):
    g = golden("rows_small")
    gen = torch.Generator().manual_seed(int(g["seed"]))
    X = torch.randn(300, 64, generator=gen)
    Y = torch.randn(280, 64, generator=gen)
    d, i = restated.knn_points(X, Y, 2, "cosine")
    assert torch.equal(i, t(g["idx"]))
    torch.testing.assert_close(d, t(g["dists"]), rtol=0, atol=1e-6)
    i1, i2, w = restated.correspondences_ratio_test(X, Y, 50)
    assert torch.equal(i1, t(g["idx1"])) and torch.equal(i2, t(g["idx2"]))
    torch.testing.assert_close(w, t(g["weight"]), rtol=0, atol=2e-6)
    torch.testing.assert_close(restated.ratio_weights(t(g["dists"])), t(g["ratio"]), rtol=0, atol=0)
    hm = t(g["heat"])
    assert torch.equal(restated.argmax_2d(hm), t(g["argmax"]))
    assert torch.equal(restated.argmax_2d(hm, max_value=False), t(g["argmin"]))
    torch.testing.assert_close(restated.pixel_grid(3, 5), t(g["grid"]), rtol=0, atol=0)


def test_spair_golden(golden, syn):
    g = golden("spair_small")
    p = syn.spair_pair(7, **SPAIR_SMALL)
    es, en, isame, inn = restated.spair_compute_errors(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"])
    torch.testing.assert_close(es, t(g["error_same"]), rtol=0, atol=1e-6)
    torch.testing.assert_close(en, t(g["error_nn"]), rtol=0, atol=1e-6)
    assert torch.equal(isame, t(g["index_same"])) and torch.equal(inn, t(g["index_nn"]))


@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
def test_restated_equals_reference_on_fresh_inputs(syn):
    ref, ref_tr = reference_loader.load()
    p = syn.scannet_pair(11, coherent=False, C=32, h=5, w=7, H=20, W=28)
    a = ref.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 64)
    b = restated.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 64)
    for x, y in zip(a, b):
        torch.testing.assert_close(x, y, rtol=0, atol=2e-6)
    p = syn.navi_pair(11, coherent=False, C=32, h=6, w=6, H=24, W=24, radius=9.0)
    a = ref.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 64)
    b = restated.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 64)
    for x, y in zip(a, b):
        torch.testing.assert_close(x, y, rtol=0, atol=2e-6)
    pts = torch.randn(9, 3)
    Rt = syn.random_rt(torch.Generator().manual_seed(3))
    torch.testing.assert_close(ref_tr.transform_points_Rt(pts, Rt), restated.transform_points_Rt(pts, Rt), rtol=0, atol=0)


@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
@pytest.mark.parametrize("kw", [dict(C=768, h=14, w=14, K=20, image_size=224), dict(C=64, h=50, w=50, K=30, image_size=800),
                                dict(C=40, h=5, w=7, K=3, image_size=64)])
def test_spair_restated_equals_the_reference_script(syn, kw):
    """the reference's own compute_errors (evaluate_spair_correspondence.py:45-103; hydra / omegaconf stubbed,
    .cuda() mapped to the identity, the model replaced by its output) against the restatement: identical."""
    for i in range(3):
        p = syn.spair_pair(30 + i, **kw)
        a = reference_loader.spair_compute_errors_reference(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"])
        b = restated.spair_compute_errors(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"], return_pred=True)
        for x, y in zip(a, b):
            assert x.shape == y.shape
            torch.testing.assert_close(x.float(), y.float(), rtol=0, atol=1e-6)
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])


@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
def test_spair_dataset_recall_and_confusion_equal_the_reference(syn):
    """evaluate_dataset of the reference script (recall + confusion matrix over a list of pairs) against the same
    quantities assembled from the restatement, the way the GPU tests assemble their expectation."""
    pairs = [syn.spair_pair(i) for i in range(6)]
    rec, conf = reference_loader.spair_evaluate_dataset_reference(pairs, 0.10)
    errs, src, tgt = [], [], []
    for p in pairs:
        es, en, isame, inn = restated.spair_compute_errors(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"])
        errs.append(es); src.append(isame); tgt.append(inn)
    errs, src, tgt = torch.cat(errs), torch.cat(src), torch.cat(tgt)
    want = torch.zeros_like(conf)
    for a, b in zip(src.tolist(), tgt.tolist()):
        want[a, b] += 1
    assert torch.equal(conf, want)
    assert abs(rec - 100.0 * (errs < 0.10).float().mean().item()) < 1e-4


def test_mutual_oracle_is_self_consistent():
    gen = torch.Generator().manual_seed(1)
    X = torch.randn(50, 16, generator=gen)
    r = restated.similarity_top2_and_mutual(X, X.clone())
    assert r["mutual"].all() and torch.equal(r["row_idx"][:, 0], torch.arange(50))


@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
def test_transformations_mirror_equals_reference(mv, syn):
    _, ref_tr = reference_loader.load()
    tr = mv.transformations
    g = torch.Generator().manual_seed(5)
    Rt = torch.stack([syn.random_rt(g) for _ in range(6)])
    pts = torch.randn(6, 17, 3, generator=g)
    assert torch.equal(tr.transform_points_Rt(pts, Rt), ref_tr.transform_points_Rt(pts, Rt))
    assert torch.equal(tr.transform_points_Rt(pts, Rt, inverse=True), ref_tr.transform_points_Rt(pts, Rt, inverse=True))
    assert torch.equal(tr.so3_rotation_angle(Rt[:, :3, :3]), ref_tr.so3_rotation_angle(Rt[:, :3, :3]))
    assert torch.equal(tr.so3_relative_angle(Rt[:3, :3, :3], Rt[3:, :3, :3]), ref_tr.so3_relative_angle(Rt[:3, :3, :3], Rt[3:, :3, :3]))
    with pytest.raises(ValueError):
        tr.so3_rotation_angle(torch.eye(3)[None] * 5)


def _navi_batch(syn, n=4, **kw):
    ps = [syn.navi_pair(40 + i, coherent=(i % 2 == 0), **kw) for i in range(n)]
    g = torch.Generator().manual_seed(77)
    Rt = torch.stack([syn.random_rt(g, max_deg=110.0) for _ in ps])  # angles spread over the four bins
    stack = lambda k: torch.stack([p[k] for p in ps])
    return stack("feat_0"), stack("feat_1"), stack("xyz_grid_0"), stack("xyz_grid_1"), Rt, stack("intrinsics")


@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
def test_navi_caller_block_restated_equals_the_reference_text(syn):
    """the reference's own evaluation loop (evaluate_navi_correspondence.py:174-221, executed from its file) against
    restated.navi_error_block fed the reference's modules: errors, the six recalls and the angle-binned recall."""
    corr, tr = reference_loader.load()
    args = _navi_batch(syn, C=32, h=6, w=6, H=24, W=24, radius=9.0)
    ref = reference_loader.navi_error_block_reference(*args, num_corr=40)
    got = restated.navi_error_block(corr, tr, *args, num_corr=40)
    assert torch.equal(ref["err_3d"], got["err_3d"]) and torch.equal(ref["err_2d"], got["err_2d"])
    want = [float(r) for r in ref["results"]]  # the script formats every number as f"{x:5.02f}"
    have = [float(f"{float(x):5.02f}") for x in list(got["recall_3d"]) + list(got["recall_2d"])]
    have += [float(f"{float(b) * 100:5.02f}") for b in got["bin_rec"]]
    assert len(want) == len(have) == 10
    for w, h in zip(want, have):
        assert (w != w and h != h) or w == h  # empty angle bins are nan in both


@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
def test_bidirectional_and_error_auc_restatements(mv):
    """the two reference entry points without a caller.  bidirectional=True: the reference's branch raises at its
    torch.cat(dim=1); its executable parts -- the two directed calls with half the budget each -- are what the
    restatement concatenates.  error_auc: restatement and product mirror against the reference's numpy."""
    corr, _ = reference_loader.load()
    gen = torch.Generator().manual_seed(12)
    X = torch.randn(120, 24, generator=gen)
    Y = X[torch.randperm(120, generator=gen)][:100] + 0.4 * torch.randn(100, 24, generator=gen)
    with pytest.raises((IndexError, RuntimeError)):
        corr.get_correspondences_ratio_test(X, Y, 30, bidirectional=True)
    a1, a2, aw = corr.get_correspondences_ratio_test(X, Y, 15)
    b2, b1, bw = corr.get_correspondences_ratio_test(Y, X, 15)
    r1, r2, rw = restated.correspondences_ratio_test_bidirectional(X, Y, 30)
    assert torch.equal(r1, torch.cat((a1, b1))) and torch.equal(r2, torch.cat((a2, b2)))
    torch.testing.assert_close(rw, torch.cat((aw, bw)), rtol=0, atol=2e-6)
    errs = [0.3, 4.0, 1.2, 9.5, 0.05, 2.2, 7.7, 3.1]
    thr = [1, 5, 10]
    want = corr.error_auc(errs, thr)
    np.testing.assert_allclose(restated.error_auc(errs, thr), want, rtol=0, atol=0)
    np.testing.assert_allclose(mv.correspondence.error_auc(errs, thr), want, rtol=0, atol=0)
    np.testing.assert_allclose(want, ERROR_AUC_GOLDEN, rtol=0, atol=1e-12)  # the constant test_host_logic checks on the GPU box



@pytest.mark.skipif(not reference_loader.available(), reason="reference tree not on this machine")
def test_adjacent_consumers_restated_equal_the_reference_text():
    """MaskCut's affinity lines and the 2AFC cosine lines, executed from the reference's files, against the restatements."""
    g = torch.Generator().manual_seed(3)
    feats = torch.rand(96, 1, generator=g) + 0.5 * torch.randn(96, 50, generator=g)
    raw, thr, d = reference_loader.maskcut_affinity_reference(feats, tau=0.6)
    A, B, dB = restated.maskcut_affinity(feats, tau=0.6)
    np.testing.assert_allclose(A.numpy(), raw, rtol=0, atol=0)
    np.testing.assert_allclose(B.numpy(), thr, rtol=0, atol=0)
    np.testing.assert_allclose(dB.numpy(), d, rtol=0, atol=1e-12)
    ref = torch.randn(20, 64, generator=g)
    left, right = ref + torch.randn(20, 64, generator=g), ref + torch.randn(20, 64, generator=g)
    a = reference_loader.twoafc_reference(ref, left, right)
    b = restated.twoafc(ref, left, right)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
