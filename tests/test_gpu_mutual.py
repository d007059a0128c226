"""Mutual matching with the two-sided ratio test (correspondence.get_mutual_correspondences, match_rows(mutual=True),
the dense helpers' mutual=True, GraphedPairMatcher(mutual=True)) against a torch restatement of its definition.

The reference has no such mode, so the definition below is the oracle: forward candidates j(i) and ratio weights
w_f(i) from each row's two best targets, reverse ones i(j), w_r(j) from each column's two best queries (both re-ranked
by 1 - cos), i mutual iff i(j(i)) == i, weight min(w_f(i), w_r(j(i))) (w_f = d0 without the ratio test), selection =
the num_corr largest weights among the mutual queries, ties to the lower query index."""
import importlib

import pytest
import torch

from oracle import restated

pytestmark = pytest.mark.gpu

GAP = 1e-3  # the north star's gap rule, applied on both sides


def mutual_oracle(P1, P2, num_corr, ratio_test=True, fp32=False):
    """fp64 throughout, or (fp32=True) the reference's arithmetic: fp64 proposes the two candidates of each side, their
    distances are fp32 1 - cosine_similarity, which re-ranks them (ties: lower index) -- on backbone features the fp32
    distances tie exactly where fp64 would still order them"""
    X = torch.nn.functional.normalize(P1.cuda().double(), dim=1)
    Y = torch.nn.functional.normalize(P2.cuda().double(), dim=1)
    S = X @ Y.t()
    fv, fi = torch.topk(S, 3, dim=1)
    rv, ri = torch.topk(S.t(), 3, dim=1)
    del S

    def weights(v):
        d = 1 - v
        return 1 - d[:, 0].clamp(min=1e-9) / d[:, 1].clamp(min=1e-9), d[:, 0]

    def rerank32(Q, T, idx):
        d = 1 - torch.nn.functional.cosine_similarity(Q[:, None, :], T[idx[:, :2]], dim=-1)
        swap = (d[:, 1] < d[:, 0]) | ((d[:, 1] == d[:, 0]) & (idx[:, 1] < idx[:, 0]))
        return torch.where(swap[:, None], d.flip(1), d), torch.where(swap[:, None], idx[:, :2].flip(1), idx[:, :2])

    if fp32:
        X32, Y32 = P1.cuda().float(), P2.cuda().float()
        dfw, fi = rerank32(X32, Y32, fi)
        drv, ri = rerank32(Y32, X32, ri)
        fv, rv = torch.cat((1 - dfw, fv[:, 2:]), 1), torch.cat((1 - drv, rv[:, 2:]), 1)
    wf_ratio, d0 = weights(fv)
    wr, _ = weights(rv)
    wf = wf_ratio if ratio_test else d0
    n = X.shape[0]
    j = fi[:, 0]
    mutual = ri[j, 0] == torch.arange(n, device=j.device)
    weight = torch.where(mutual, torch.minimum(wf, wr[j]) if ratio_test else wf, torch.full_like(wf, -float("inf")))
    gap = (fv[:, 0] - fv[:, 1] > GAP) & (rv[j, 0] - rv[j, 1] > GAP)
    # a ratio weight also depends on WHICH row is second: where the second and third similarities are within the product's
    # rounding, the tensor cores may propose the third, and the weight moves by up to that difference
    gap2 = gap & (fv[:, 1] - fv[:, 2] > GAP) & (rv[j, 1] - rv[j, 2] > GAP)
    order = torch.sort(-weight, stable=True).indices  # ties: lower query index
    k = min(num_corr, int(mutual.sum()))
    sel = order[:k]
    return {"j": j, "wf": wf, "wr": wr, "mutual": mutual, "weight": weight, "gap": gap, "gap2": gap2, "sel": sel, "sel_dst": j[sel],
            "sel_w": weight[sel]}


def run_lib(C_, P1, P2, num_corr, ratio_test=True):
    dev = torch.device("cuda")
    (A16, A32), (B16, B32), mu = C_._rows_pair(P1, P2, dev)
    r = C_.match_rows(A16, A32, B16, B32, P1.shape[0], P2.shape[0], num_corr, ratio_test, center_B=mu, mutual=True)
    torch.cuda.synchronize()
    return r


def gaussian(n, m, C, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, C, generator=g), torch.randn(m, C, generator=g)


@pytest.fixture
def precision(mv):
    saved = mv.correspondence.set_match_precision()
    yield mv.correspondence.set_match_precision
    mv.correspondence._CFG.update(saved)


SHAPES = {"navi": (5024, 5024, 3072), "scannet": (18231, 18231, 2048)}


@pytest.mark.parametrize("shape", ["navi", "scannet"])
@pytest.mark.parametrize("dtype", ["f16", "bf16", "tf32"])
@pytest.mark.parametrize("ratio_test", [True, False])
def test_mutual_gaussian_maps(mv, precision, shape, dtype, ratio_test):
    precision(dtype=dtype)
    C_ = mv.correspondence
    n, m, C = SHAPES[shape]
    P1, P2 = gaussian(n, m, C, 17)
    o = mutual_oracle(P1, P2, 1000, ratio_test)
    r = run_lib(C_, P1, P2, 1000, ratio_test)
    gap, gap2 = o["gap"], o["gap2"]
    frac, frac2 = float(gap.float().mean()), float(gap2.float().mean())
    print(f"{shape} {dtype} ratio_test={ratio_test}: gap set {100 * frac:.1f} % of the queries ({100 * frac2:.1f} % with the "
          f"second-third gaps too), {int(o['mutual'].sum())} mutual")
    assert frac > 0.3 and frac2 > 0.15
    assert torch.equal(r.row_idx[:, 0].long()[gap], o["j"][gap])
    assert torch.equal(r.mutual_rr.bool()[gap], o["mutual"][gap])
    jg = o["j"][gap]
    assert torch.equal(r.col_idx[jg, 0].long() == torch.arange(n, device=jg.device)[gap], o["mutual"][gap])
    # both weights where both neighbours of both sides are clear
    j2 = o["j"][gap2]
    assert (r.weight.double()[gap2] - o["wf"][gap2]).abs().max() <= 1e-6
    assert (r.col_weight.double()[j2] - o["wr"][j2]).abs().max() <= 1e-6
    # the selection: mutual queries only, sorted, and the oracle's set
    k = int(r.k_dev.item())
    assert k == min(1000, int(r.mutual_rr.sum()))
    src = r.sel_src[:k].long()
    assert bool(r.mutual_rr[src].bool().all())
    assert bool((r.sel_weight[:k][1:] <= r.sel_weight[:k][:-1]).all())
    shared = len(set(src.tolist()) & set(o["sel"].tolist()))
    assert shared >= 0.99 * max(len(o["sel"]), 1), (shared, len(o["sel"]))
    # the public helper returns the same selection
    i1, i2, w = C_.get_mutual_correspondences(P1, P2, 1000, ratio_test=ratio_test)
    assert i1.device.type == "cpu" and torch.equal(i1, src.cpu()) and torch.equal(i2, r.sel_dst[:k].long().cpu())
    assert torch.equal(w, r.sel_weight[:k].cpu())


def test_mutual_symmetry(mv):
    C_ = mv.correspondence
    P1, P2 = gaussian(5024, 4000, 768, 3)
    o = mutual_oracle(P1, P2, 1000)
    r12 = run_lib(C_, P1, P2, 1000)
    r21 = run_lib(C_, P2, P1, 1000)
    gap = o["gap"]
    # (i, j) mutual in (P1, P2) <=> (j, i) mutual in (P2, P1), on the queries whose decision is clear
    i = torch.arange(P1.shape[0], device="cuda")[gap]
    j = r12.row_idx[gap, 0].long()
    fwd = r12.mutual_rr.bool()[gap]
    rev = r21.mutual_rr.bool()[j] & (r21.row_idx[j, 0].long() == i)
    assert torch.equal(fwd, rev)
    j2 = r12.row_idx[o["gap2"], 0].long()
    assert (r12.col_weight[j2] - r21.weight[j2]).abs().max() <= 1e-6


def test_mutual_ties_go_to_the_lower_index(mv):
    C_ = mv.correspondence
    P1, P2 = gaussian(600, 500, 64, 9)
    P1[400] = P1[7]  # duplicated query: only the lower one can be its column's best
    P2[300] = P2[20]  # duplicated target: every query prefers the lower one
    r = run_lib(C_, P1, P2, 600)
    assert not bool((r.row_idx[:, 0] == 300).any())
    assert r.mutual_rr[400] == 0


def test_mutual_false_is_todays_call(mv):
    C_ = mv.correspondence
    p = importlib.import_module("midvision-probe_b200.synthetic").navi_pair(0, C=256, h=14, w=14, H=56, W=56)
    a = C_.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 300)
    b = C_.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 300, mutual=False)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


# ---- the dense helpers on backbone features ----------------------------------------------------------------------
NAVI_THR3, SCAN_THR3 = [0.01, 0.02, 0.05], [0.01, 0.02, 0.05, 0.10]


@pytest.fixture(scope="module")
def bb():
    return importlib.import_module("midvision-probe_b200.backbones")


def _pair(bb, kind, seed, model):
    if kind == "navi":
        p = bb.navi_backbone_pair(seed, model, device="cuda", noise=0.7)
        x0, f0, _, _ = restated.xyz_side(p["feat_0"], p["xyz_grid_0"])
        x1, f1, _, _ = restated.xyz_side(p["feat_1"], p["xyz_grid_1"])
        return p, x0, f0, x1, f1, p["intrinsics"]
    p = bb.scannet_backbone_pair(seed, model, device="cuda", noise=1.0)
    x0, f0, _ = restated.depth_side(p["feat_0"], p["depth_0"], p["K"])
    x1, f1, _ = restated.depth_side(p["feat_1"], p["depth_1"], p["K"])
    return p, x0, f0, x1, f1, p["K"]


def _helper(C_, kind, p):
    if kind == "navi":
        return C_.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 1000, mutual=True)
    return C_.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 1000, mutual=True)


def _keyset(a, b):
    return {tuple(u.tolist()) + tuple(v.tolist()) for u, v in zip(a.cpu(), b.cpu())}


# NAVI-shaped ViT features: the selections share >= 990 of 1000 (of k) and recall is within 0.1 pp.  ScanNet-shaped ResNet
# features (near-collinear, mean pixel cosine ~0.93): measured 945, 999, 999 and 838 of 937 shared over the four seeds -- the
# mutual decision i(j(i)) == i flips wherever a column's best rows are within rounding of each other -- so there the rule is
# applied to the selected queries whose forward AND reverse top-2 gaps exceed 1e-3, and recall is reported, not gated.


@pytest.mark.parametrize("kind", ["navi", "scannet"])
@pytest.mark.parametrize("graphs", [1, 0])
def test_mutual_dense_helpers_on_backbone_features(mv, bb, precision, kind, graphs):
    C_ = mv.correspondence
    precision(helper_graphs=graphs)
    model = (bb.DenseViT(bb.vit_b16(0, img_size=224), multilayer=True) if kind == "navi" else bb.resnet50_layer4(0)).cuda()
    thr = NAVI_THR3 if kind == "navi" else SCAN_THR3
    hits_lib, hits_ref, tot_lib, tot_ref = torch.zeros(len(thr)), torch.zeros(len(thr)), 0, 0
    for seed in range(4):
        p, x0, f0, x1, f1, Kmat = _pair(bb, kind, seed, model)
        o = mutual_oracle(f0, f1, 1000, fp32=True)
        got = _helper(C_, kind, p)
        ref0, ref1 = x0.cuda()[o["sel"]], x1.cuda()[o["sel_dst"]]
        k = got[0].shape[0]
        shared = len(_keyset(got[0], got[1]) & _keyset(ref0, ref1))
        print(kind, "seed", seed, "shared", shared, "of", k, len(o["sel"]))
        if kind == "navi":
            assert shared >= 0.99 * max(min(k, len(o["sel"])), 1), (seed, shared, k, len(o["sel"]))
        else:
            clear = o["gap"][o["sel"]]
            want = _keyset(ref0[clear], ref1[clear])
            got_clear = len(_keyset(got[0], got[1]) & want)
            print(kind, "seed", seed, "clear", len(want), "shared", got_clear)
            assert got_clear >= 0.99 * len(want), (seed, got_clear, len(want))
        e3, _ = restated.pair_errors(got[0].cpu(), got[1].cpu(), p["Rt"], Kmat)
        r3, _ = restated.pair_errors(ref0.cpu(), ref1.cpu(), p["Rt"], Kmat)
        hits_lib += torch.tensor([float((e3 < t).sum()) for t in thr])
        hits_ref += torch.tensor([float((r3 < t).sum()) for t in thr])
        tot_lib += len(e3)
        tot_ref += len(r3)
    rec_lib, rec_ref = 100 * hits_lib / max(tot_lib, 1), 100 * hits_ref / max(tot_ref, 1)
    print(kind, "recall", rec_lib.tolist(), "oracle", rec_ref.tolist(), "k", tot_lib, tot_ref)
    if kind == "navi":
        assert (rec_lib - rec_ref).abs().max() <= 0.1


def test_mutual_lowrank_routes_agree(mv, bb, precision):
    """ScanNet shape: the low-rank route forced on and off selects the same matches on the gap set."""
    C_ = mv.correspondence
    model = bb.resnet50_layer4(0).cuda()
    p, x0, f0, x1, f1, _ = _pair(bb, "scannet", 1, model)
    o = mutual_oracle(f0, f1, 1000)
    clear = o["gap"][o["sel"]]
    want = _keyset(x0.cuda()[o["sel"]][clear], x1.cuda()[o["sel_dst"]][clear])
    sets = []
    for lowrank in ("1", "0"):
        precision(lowrank=lowrank, helper_graphs=0)
        got = _helper(C_, "scannet", p)
        sets.append(_keyset(got[0], got[1]) & want)
    assert sets[0] == sets[1]


@pytest.mark.parametrize("kind", ["navi", "scannet"])
def test_mutual_graphed_matcher_counts(mv, bb, kind):
    """GraphedPairMatcher(mutual=True), single graph, scores the ungraphed call's counts."""
    ev = importlib.import_module("midvision-probe_b200.evaluation")
    model = (bb.DenseViT(bb.vit_b16(0, img_size=224), multilayer=True) if kind == "navi" else bb.resnet50_layer4(0)).cuda()
    p, *_ = _pair(bb, kind, 2, model)
    thr3, thr2 = [0.01, 0.05], [5, 25]
    acc_g = ev.RecallAccumulator(thr3, thr2, device=torch.device("cuda"))
    acc_e = ev.RecallAccumulator(thr3, thr2, device=torch.device("cuda"))
    if kind == "navi":
        gm = ev.GraphedPairMatcher("xyz", tuple(p["feat_0"].shape), tuple(p["xyz_grid_0"].shape), 1000, mutual=True).capture()
        gm.load(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"])
        gm.run(acc_g, p["Rt"], p["intrinsics"])
        K = p["intrinsics"]
    else:
        gm = ev.GraphedPairMatcher("depth", tuple(p["feat_0"].shape), tuple(p["depth_0"].shape), 1000, K=p["K"], mutual=True).capture()
        gm.load(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"])
        gm.run(acc_g, p["Rt"])
        K = p["K"]
    torch.cuda.synchronize()
    r = gm.out[2]
    assert int(r.k_dev.item()) <= r.k
    # ungraphed: the same pipeline body, launched eagerly
    s0, s1, r_e = gm._body()
    acc_e.score(r_e, s0.xyz, s1.xyz, p["Rt"], K)
    torch.cuda.synchronize()
    assert torch.equal(acc_g.hits, acc_e.hits)
    assert int(r_e.k_dev.item()) == int(r.k_dev.item())
