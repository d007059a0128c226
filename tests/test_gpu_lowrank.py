"""The low-rank proposal operands of kernel 2 (csrc/lr_gram.cu): the product of the fp16 operand rows over the target
image's SOURCE PIXELS must reproduce the cosine similarity of the reference's interpolated, normalised rows
(correspondence.py:164-176 / :240-241 + :47-48), most precisely where a row's best columns are; and the dense helpers must
return the reference's matches when kernel 2 ranks that product instead of the C-channel one."""
import importlib

import pytest
import torch
import torch.nn.functional as F

from oracle import restated

pytestmark = pytest.mark.gpu


@pytest.fixture()
def lowrank_on(mv):
    C_ = mv.correspondence
    C_.set_match_precision(lowrank=1)
    yield
    C_.set_match_precision(lowrank="auto")


def sides(mv, kind, p):
    C_ = mv.correspondence
    L = mv._lib
    dev = torch.device("cuda")
    if kind == "depth":
        Kc = p["K"].float()
        Kh, Kinv = C_._host_mat(Kc), C_._host_mat(Kc.inverse())
        s0 = C_.prepare_depth_side(p["feat_0"].cuda(), p["depth_0"], Kh, Kinv, dev)
        s1 = C_.prepare_depth_side(p["feat_1"].cuda(), p["depth_1"], Kh, Kinv, dev)
        f0 = restated.depth_side(p["feat_0"], p["depth_0"], p["K"])[1]
        f1 = restated.depth_side(p["feat_1"], p["depth_1"], p["K"])[1]
    else:
        s0 = C_.prepare_xyz_side(p["feat_0"].cuda(), p["xyz_grid_0"], dev)
        s1 = C_.prepare_xyz_side(p["feat_1"].cuda(), p["xyz_grid_1"], dev)
        f0 = restated.xyz_side(p["feat_0"], p["xyz_grid_0"])[1]
        f1 = restated.xyz_side(p["feat_1"], p["xyz_grid_1"])[1]
    return s0, s1, f0, f1


@pytest.mark.parametrize("kind,shape", [("depth", dict(C=256, h=15, w=20, H=60, W=80)), ("depth", dict(C=64, h=7, w=9, H=40, W=52)),
                                        ("xyz", dict(C=256, h=14, w=14, H=56, W=56, radius=22.0)),
                                        ("xyz", dict(C=128, h=9, w=11, H=36, W=44, radius=15.0)),
                                        # every width of lr_build_query (KT = ceil(hwp / 64) -> 8, 13, 16) up to the 1024-pixel limit.  The
                                        # top-2 error is the fp16 rounding of A - c_i at the best candidates' taps; it does not depend on the
                                        # width (an fp16 emulation of the operands gives the same 1.2-1.6e-4 at 14 x 14 and 32 x 32, C = 256)
                                        # but on how far those taps sit below the row's maximum: it grows with sparse targets (a 1.3x
                                        # upsample or 90 % of the pixels invalid: 2-3e-4) and, for the 16 bicubic taps (sum |B| ~ 2.8), with
                                        # the 1 / sqrt(C) spread of the cosines between Gaussian features (C = 128: 2.4e-4 at 28 x 28,
                                        # 1.6e-4 already at 14 x 14).  So these shapes keep the regime of the ones above: a dense 4x upsample,
                                        # C = 256 for the bicubic ones
                                        ("depth", dict(C=256, h=18, w=20, H=36, W=40)), ("xyz", dict(C=256, h=16, w=21, H=32, W=42, radius=30.0)),
                                        ("depth", dict(C=256, h=24, w=24, H=96, W=96)), ("xyz", dict(C=256, h=28, w=28, H=112, W=112, radius=50.0)),
                                        ("depth", dict(C=128, h=30, w=30, H=120, W=120)), ("xyz", dict(C=256, h=32, w=32, H=128, W=128, radius=56.0))])
@pytest.mark.parametrize("exact", [False, True])
def test_operand_product_equals_the_cosine_similarity(mv, syn, kind, shape, exact):
    """exact=False: cosine Gram of fp16 unit rows from kernel 2; exact=True: fp32 Gram of the raw rows from the CUDA cores"""
    C_ = mv.correspondence
    p = syn.scannet_pair(3, **shape) if kind == "depth" else syn.navi_pair(3, **shape)
    s0, s1, f0, f1 = sides(mv, kind, p)
    n, m = f0.shape[0], f1.shape[0]
    assert (s0.n, s1.n) == (n, m)
    A, B, K = C_._lowrank_operands(s0, s1, n, m, None, None, exact=exact)[:3]
    torch.cuda.synchronize()
    h, w = shape["h"], shape["w"]
    hw = h * w
    hwp = (hw + 7) // 8 * 8
    assert K == hwp + 8
    A, B = A[:, :K].double(), B[:, :K].double()  # fp64 on the device: the widest shapes have ~15k points per side
    S = A @ B.t()
    a, b = F.normalize(f0, dim=-1).double().cuda(), F.normalize(f1, dim=-1).double().cuda()
    S_ref = a @ b.t()
    err = (S - S_ref).abs()
    # fp16 operands: 2^-11 relative on entries of magnitude <= 1, a handful of terms per product
    assert err.max() < 2e-3, float(err.max())
    # ... and far better where it matters: at every row's two best columns (the row is centred on its maximum)
    top = torch.topk(S_ref, 2, dim=1).indices
    assert err.gather(1, top).max() < 2e-4, float(err.gather(1, top).max())
    # structure: a target row has at most 4 (bilinear) / 16 (bicubic) non-zeros among the source-pixel columns, zeros in the
    # padding, and two augmentation columns that add up to the row sum; a query row's augmentation columns repeat its centre
    nnz = (B[:, :hwp] != 0).sum(1)
    assert int(nnz.max()) <= (4 if kind == "depth" else 16)
    assert (B[:, hw:hwp] == 0).all() and (A[:, hw:hwp] == 0).all()
    assert ((B[:, hwp] + B[:, hwp + 1]) - B[:, :hw].sum(1)).abs().max() < 2e-3
    assert torch.equal(A[:, hwp], A[:, hwp + 1]) and (A[:, hwp + 2:] == 0).all() and (B[:, hwp + 2:] == 0).all()
    assert (A[:, :hw].max(1).values.abs() < 1e-3).all()  # centred on the row maximum


@pytest.mark.parametrize("kind", ["depth", "xyz"])
def test_helpers_with_the_lowrank_proposal_match_the_oracle(mv, syn, lowrank_on, kind):
    """small pairs through the public helpers with the low-rank proposal forced on: the reference's matches"""
    C_ = mv.correspondence
    for seed in range(3):
        if kind == "depth":
            p = syn.scannet_pair(seed, C=256, h=15, w=20, H=60, W=80)
            got = C_.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 500)
            ref = restated.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 500)
        else:
            p = syn.navi_pair(seed, C=256, h=14, w=14, H=56, W=56, radius=22.0)
            got = C_.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 500)
            ref = restated.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 500)
        gset = {tuple(a.tolist()) + tuple(b.tolist()) for a, b in zip(got[0].cpu(), got[1].cpu())}
        rset = {tuple(a.tolist()) + tuple(b.tolist()) for a, b in zip(ref[0], ref[1])}
        assert len(gset & rset) >= 495, (kind, seed, len(gset & rset))
        # the ratio weights of the selected matches: equal, except where a row's SECOND candidate is a near-tie of the
        # third (the weight then moves by that gap; the match itself is the same)
        diff = (torch.sort(got[2].cpu()).values - torch.sort(ref[2]).values).abs()
        assert int((diff > 2e-5).sum()) <= 5 and float(diff.max()) < 5e-3, (kind, seed, float(diff.max()))


@pytest.mark.parametrize("C,h,w,taps", [(2048, 15, 20, 2), (256, 9, 7, 4), (3072, 12, 12, 4), (320, 28, 28, 2),
                                         (128, 32, 32, 4), (256, 31, 33, 2)])  # off1 = 1024: the limit
def test_exact_gram_is_fp32_exact(mv, C, h, w, taps):
    """mv_lr_gram_exact against an fp64 product: every entry it promises (the whole cross block, the same-image entries whose
    indices are at most `reach` apart) to ~1 ulp (blocked fp32 accumulation), symmetric, pad rows zero, snorm / rsnorm from
    the diagonal; bit-repeatable."""
    L, C_ = mv._lib, mv.correspondence
    g = torch.Generator().manual_seed(C + h)
    hw = h * w
    off1 = (hw + 31) // 32 * 32
    reach = (taps - 1) * (w + 1)
    # all-positive, nearly collinear rows (the CNN regime) and signed rows
    s0 = (torch.rand(hw, C, generator=g) + 0.5).cuda()
    s1 = torch.randn(hw, C, generator=g).cuda()
    outs = []
    for _ in range(2):
        G = torch.full((2 * off1, 2 * off1), 7.0, device="cuda")
        sn = torch.empty(2 * off1, device="cuda")
        rs = torch.empty(2 * off1, device="cuda")
        L.call("mv_lr_gram_exact", L.ptr(s0), L.ptr(s1), C, hw, off1, reach, L.ptr(G), 2 * off1, L.ptr(sn), L.ptr(rs), C_._stream())
        torch.cuda.synchronize()
        outs.append(G)
    assert torch.equal(outs[0], outs[1])
    G = outs[0]
    R = torch.zeros(2 * off1, C, dtype=torch.float64, device="cuda")
    R[:hw] = s0.double()
    R[off1:off1 + hw] = s1.double()
    ref = R @ R.t()
    scale = (R.norm(dim=1)[:, None] * R.norm(dim=1)[None, :]).clamp_min(1e-30)
    idx = torch.arange(2 * off1, device="cuda")
    same_img = (idx[:, None] < off1) == (idx[None, :] < off1)
    promised = ~same_img | ((idx[:, None] - idx[None, :]).abs() <= reach)
    rel = ((G.double() - ref).abs() / scale)[promised]
    assert float(rel.max()) < 2.5e-7, float(rel.max())   # relative to |a||b|: a few ulp of a cosine
    assert torch.equal(torch.where(promised, G, 0), torch.where(promised, G.t(), 0))
    pad = torch.ones(2 * off1, dtype=torch.bool, device="cuda")
    pad[:hw] = False
    pad[off1:off1 + hw] = False
    assert (G[pad][:, ~pad][promised[pad][:, ~pad]] == 0).all()
    torch.testing.assert_close(sn.double(), R.norm(dim=1), rtol=3e-7, atol=0)
    assert (rs[pad] == 0).all()


@pytest.mark.parametrize("kind", ["depth", "xyz"])
def test_k3_on_the_gram_matrix_equals_the_oracle_distances(mv, syn, kind):
    """mv_k3_ratio_mutual_lr: the fp32 cosine distances of the two candidates from the Gram matrix against the reference's own
    1 - cosine_similarity of the gathered rows (correspondence.py:53-58): <= 1e-6, same neighbours, same weights."""
    C_ = mv.correspondence
    shape = dict(C=256, h=15, w=20, H=60, W=80) if kind == "depth" else dict(C=256, h=14, w=14, H=56, W=56, radius=22.0)
    p = syn.scannet_pair(4, **shape) if kind == "depth" else syn.navi_pair(4, **shape)
    s0, s1, f0, f1 = sides(mv, kind, p)
    s0.rows16 = s0.rows32 = s0.rows_lo = s1.rows16 = s1.rows32 = s1.rows_lo = None   # as prepared with want_rows=False
    r = C_._match_sides(s0, s1, s0.n, s1.n, 500)
    torch.cuda.synchronize()
    d_ref, i_ref = restated.knn_points(f0, f1, 2, "cosine")
    o = restated.similarity_top2_and_mutual(f0, f1)
    clear = o["row_gap"] > 1e-3
    idx = r.row_idx.cpu().long()
    assert torch.equal(idx[clear, 0], i_ref[clear, 0])
    same = (idx == i_ref).all(1)
    assert float(same.float().mean()) > 0.9
    assert float((r.dists.cpu()[same] - d_ref[same]).abs().max()) <= 1e-6
    w_ref = restated.ratio_weights(d_ref)
    assert float((r.weight.cpu()[same] - w_ref[same]).abs().max()) <= 2e-5


def test_lowrank_is_the_default_where_it_pays(mv):
    C_ = mv.correspondence
    assert C_._CFG["lowrank"] == "auto"
    assert C_.lowrank_applies(2048, 15, 20, 19200, 19200)            # ScanNet-shaped: 312 columns instead of 2056
    assert not C_.lowrank_applies(3072, 28, 28, 12544, 12544)        # NAVI-shaped: the dense product stays
    assert not C_.lowrank_applies(768, 14, 14, 196, 20)              # small problems
    assert C_.lowrank_exact_applies(2048, 15, 20, 19200, 19200)      # ... and there without kernel 1 (kernel 3 on the exact Gram)


def test_full_size_scannet_pair_same_result_with_and_without(mv, syn):
    """ScanNet-shaped Gaussian pair at full size: the default (low-rank proposal) and the C-channel product give the same
    selected matches (up to ties: >= 995 of 1000) and the helper's neighbour indices agree wherever the reference gap is clear."""
    C_ = mv.correspondence
    p = syn.scannet_pair(5)
    out = {}
    for name, lr, k3 in (("exact", "auto", 1), ("rows", "auto", 0), ("dense", 0, 1)):
        C_.set_match_precision(lowrank=lr, lowrank_k3=k3)
        try:
            out[name] = C_.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 1000)
        finally:
            C_.set_match_precision(lowrank="auto", lowrank_k3=1)
    sets = {k: {tuple(x.tolist()) + tuple(y.tolist()) for x, y in zip(v[0].cpu(), v[1].cpu())} for k, v in out.items()}
    assert len(sets["exact"] & sets["dense"]) >= 995, len(sets["exact"] & sets["dense"])
    assert len(sets["rows"] & sets["dense"]) >= 995, len(sets["rows"] & sets["dense"])
    # north-star rule on the proposal itself: the nearest neighbour of every row whose reference fp32 top-2 gap exceeds 1e-3
    s0, s1, f0, f1 = sides(mv, "depth", p)
    assert C_.lowrank_applies(*s0.fshape, s0.n, s1.n, s0.mode)
    r = C_._match_sides(s0, s1, s0.n, s1.n, 1000)
    o = restated.similarity_top2_and_mutual(f0, f1)
    clear = o["row_gap"] > 1e-3
    assert float(clear.float().mean()) > 0.5
    assert torch.equal(r.row_idx[:, 0].cpu().long()[clear], o["row_idx"][clear, 0])
    cclear = o["col_gap"] > 1e-3  # and the mutual flag wherever both the row's and its column's decision are clear
    both = clear & cclear[o["row_idx"][:, 0]]
    assert torch.equal(r.mutual.cpu().bool()[both], o["mutual"][both])


@pytest.mark.parametrize("kind", ["xyz", "depth"])
@pytest.mark.parametrize("split", [False, True])
def test_lowrank_graph_replay_equals_eager(mv, syn, lowrank_on, kind, split):
    """the exact low-rank route inside the captured CUDA graphs (one graph, and the split target / query pair of graphs the
    synchronous helper replays; device-resident live counts) gives the integer counts and the selected matches of the eager
    launches with host-known counts, pair after pair."""
    ev = mv.evaluation
    thr3, thr2 = [0.01, 0.02, 0.05], [5.0, 25.0, 50.0]
    if kind == "xyz":
        pairs = [syn.navi_pair(i, C=256, h=14, w=14, H=56, W=56, radius=20.0) for i in range(3)]
        gk = ("xyz_grid_0", "xyz_grid_1", "intrinsics")
    else:
        pairs = [syn.scannet_pair(i, C=256, h=15, w=21, H=60, W=84) for i in range(3)]  # 315 source pixels: not a multiple of 8
        gk = ("depth_0", "depth_1", "K")
    gm = ev.GraphedPairMatcher(kind, tuple(pairs[0]["feat_0"].shape), tuple(pairs[0][gk[0]].shape), 300, K=pairs[0].get("K"),
                               split=split).capture()
    assert gm.lowrank_exact
    for p in pairs + pairs[:1]:
        a = ev.RecallAccumulator(thr3, thr2, device="cuda")
        b = ev.RecallAccumulator(thr3, thr2, device="cuda")
        gm.load(p["feat_0"], p["feat_1"], p[gk[0]], p[gk[1]])
        rg = gm.run(a, p["Rt"], p[gk[2]])
        if kind == "xyz":
            re_ = ev.match_and_score_xyz(p["feat_0"], p["feat_1"], p[gk[0]], p[gk[1]], p[gk[2]], p["Rt"], 300, b, sync=True)
        else:
            re_ = ev.match_and_score_depth(p["feat_0"], p["feat_1"], p[gk[0]], p[gk[1]], p[gk[2]], p["Rt"], 300, b, sync=True)
        assert a.hits.cpu().tolist() == b.hits.cpu().tolist()
        k = re_.k
        assert int(rg.k_dev.item()) == k
        assert torch.equal(rg.sel_src[:k], re_.sel_src[:k]) and torch.equal(rg.sel_weight[:k], re_.sel_weight[:k])


def test_lowrank_with_few_live_points_and_border_taps(mv, syn, lowrank_on):
    """mostly empty depth maps (a few hundred live points, many of them at the image border where bilinear taps fall outside
    the map and are dropped) through the low-rank route: the reference's matches."""
    C_ = mv.correspondence
    for seed in range(2):
        p = syn.scannet_pair(10 + seed, C=128, h=8, w=10, H=48, W=60, zero_frac=0.9)
        got = C_.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 100)
        ref = restated.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 100)
        gset = {tuple(a.tolist()) + tuple(b.tolist()) for a, b in zip(got[0].cpu(), got[1].cpu())}
        rset = {tuple(a.tolist()) + tuple(b.tolist()) for a, b in zip(ref[0], ref[1])}
        assert got[0].shape == ref[0].shape
        assert len(gset & rset) >= int(0.97 * len(rset)), (seed, len(gset & rset), len(rset))
