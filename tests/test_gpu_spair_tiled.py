"""The tiled form of the SPair batch match (mv_spair_match_batch_tiled), which compute_errors_batch takes for maps above
256 pixels: 50 x 50 and 57 x 57 at the reference's 800-pixel input, stride-32 CNN maps, key-point tiles, odd and
non-square maps, partial pixel tiles.  Checked against the oracle (fp32 torch on the CPU) pair by pair, against the first
form, for 16-bit bit identity, batch independence, repeatability and graph capture."""
import importlib
from ctypes import c_float

import pytest
import torch

from oracle import restated

pytestmark = pytest.mark.gpu

DTYPES = [torch.bfloat16, torch.float16]


def batch(syn, seed, B, C, h, w, K, image_size):
    pairs = [syn.spair_pair(seed + i, C=C, h=h, w=w, K=K, image_size=image_size) for i in range(B)]
    return (torch.stack([p["feats"] for p in pairs]), torch.stack([p["kps_i"] for p in pairs]),
            torch.stack([p["kps_j"] for p in pairs]), [p["thresh_scale"] for p in pairs], image_size)


def run(mv, feats, ki, kj, ts, size, kp_max=64):
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")
    conf = torch.zeros((kp_max, kp_max), dtype=torch.int64, device="cuda")
    out = mv.spair.compute_errors_batch(feats, ki, kj, ts, size, hits=hits, confusion=conf)
    return tuple(x.cpu() for x in out) + (hits.cpu(), conf.cpu())


def first_form(mv, feats, ki, kj, ts, size, kp_max=64):
    """the same batch through mv_spair_match_batch (fp32): the one-CTA-per-pair first form at these sizes."""
    L = mv._lib
    f = feats.float().cuda().contiguous()
    B, _, C, h, w = f.shape
    K = ki.shape[1]
    ki, kj = ki.float().cuda().contiguous(), kj.float().cuda().contiguous()
    t = torch.as_tensor(ts, dtype=torch.float32).cuda()
    pred = torch.empty((B, K), dtype=torch.int32, device="cuda")
    es = torch.empty((B, K), dtype=torch.float32, device="cuda")
    en = torch.empty_like(es)
    inn = torch.empty_like(pred)
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")
    conf = torch.zeros((kp_max, kp_max), dtype=torch.int64, device="cuda")
    L.call("mv_spair_match_batch", L.ptr(f), B, C, h, w, L.ptr(ki), L.ptr(kj), K, ki.shape[2], L.ptr(t), c_float(float(size)),
           c_float(0.10), L.ptr(pred), L.ptr(es), L.ptr(en), L.ptr(inn), L.ptr(hits), L.ptr(conf), kp_max,
           mv.correspondence._stream())
    return tuple(x.cpu() for x in (es, en, inn, pred, hits, conf))


def check_oracle(mv, feats, ki, kj, ts, size, gap=1e-5):
    """per pair: arg-max identical wherever the oracle's top-2 gap exceeds `gap`, key points kept bit-exact, errors to 1e-5;
    hits equal to the oracle's counts; confusion exact for clear pairs, the kernel's index_nn for pairs with a near-tie."""
    B, K = ki.shape[0], ki.shape[1]
    es, en, inn, pred, hits, conf = run(mv, feats, ki, kj, ts, size, kp_max=K)
    inn, pred = inn.long(), pred.long()
    want_conf = torch.zeros((K, K), dtype=torch.int64)
    n_both = n_hit = unclear = 0
    for b in range(B):
        oes, oen, oisame, oinn, heat = restated.spair_compute_errors(feats[b].float(), ki[b], kj[b], ts[b], size, return_pred=True)
        flat = heat.flatten(1)
        top2 = torch.topk(flat, 2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > gap
        unclear += int((~clear).sum())
        assert torch.equal(pred[b][clear], flat.argmax(1)[clear]), b
        assert torch.equal((es[b] >= 0).nonzero().squeeze(1), oisame)
        ok = clear[oisame]
        torch.testing.assert_close(es[b][oisame][ok], oes[ok], rtol=0, atol=1e-5)
        if bool(clear.all()):
            torch.testing.assert_close(en[b][oisame], oen, rtol=0, atol=1e-5)
            assert torch.equal(inn[b][oisame], oinn)
            pairs_nn = zip(oisame.tolist(), oinn.tolist())
        else:
            pairs_nn = zip(oisame.tolist(), inn[b][oisame].tolist())
        for a_, b_ in pairs_nn:
            want_conf[a_, b_] += 1
        n_both += oisame.numel()
        n_hit += int((es[b][oisame] < 0.10).sum())
    assert unclear <= max(B, B * K // 20)
    assert hits.tolist() == [n_both, n_hit]
    assert torch.equal(conf, want_conf)


def assert_same_bits(a, b):
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and x.shape == y.shape
        xb = x.view(torch.int32) if x.dtype == torch.float32 else x
        yb = y.view(torch.int32) if y.dtype == torch.float32 else y
        assert torch.equal(xb, yb), int((xb != yb).sum())


SHAPES = [dict(C=768, h=50, w=50, K=30, image_size=800, B=3),   # ViT-B/16 at 800 px
          dict(C=768, h=57, w=57, K=30, image_size=800, B=2),   # ViT/14 at 800 px: odd h*w
          dict(C=768, h=28, w=28, K=20, image_size=448, B=3),
          dict(C=2048, h=25, w=25, K=30, image_size=800, B=2),  # stride-32 CNN: two key-point tiles in the first form
          dict(C=64, h=16, w=17, K=20, image_size=272, B=4),    # 272 pixels: just above 256, a 16-pixel last tile
          dict(C=104, h=17, w=19, K=17, image_size=320, B=3),   # odd h*w, a tail channel chunk
          dict(C=96, h=20, w=30, K=12, image_size=480, B=3)]    # not square, 88-pixel last tile


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s['C']}x{s['h']}x{s['w']}K{s['K']}")
def test_against_oracle(mv, syn, shape):
    s = dict(shape)
    B = s.pop("B")
    check_oracle(mv, *batch(syn, 3000, B, **s))


@pytest.mark.parametrize("K", [1, 8, 20, 30, 33, 64])
def test_keypoint_counts(mv, syn, K):
    check_oracle(mv, *batch(syn, 3100 + K, 3, C=64, h=21, w=23, K=K, image_size=336))


def test_single_tf32_term(mv, syn):
    prev = mv.spair.set_heatmap_precision("tf32")
    try:
        check_oracle(mv, *batch(syn, 3200, 3, C=768, h=50, w=50, K=30, image_size=800), gap=1e-3)
    finally:
        mv.spair.set_heatmap_precision(prev)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("hw", [(50, 50), (57, 57)])
def test_16bit_bit_identical_to_widened(mv, syn, dtype, precision, hw):
    feats, ki, kj, ts, size = batch(syn, 3300, 3, C=768, h=hw[0], w=hw[1], K=30, image_size=800)
    f16 = feats.to(dtype).cuda()
    prev = mv.spair.set_heatmap_precision(precision)
    try:
        a = run(mv, f16, ki, kj, ts, size)
        b = run(mv, f16.float(), ki, kj, ts, size)
    finally:
        mv.spair.set_heatmap_precision(prev)
    assert_same_bits(a, b)
    assert int(a[4][0]) > 0


def test_batch_independence_and_repeatability(mv, syn):
    """more work units than resident CTAs; each pair alone gives the bits it gets inside the large batch; two calls agree."""
    distinct = 7
    feats, ki, kj, ts, size = batch(syn, 3400, distinct, C=64, h=50, w=50, K=30, image_size=800)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    B = (2 * sm) // 10 * 3 + 5   # 10 pixel tiles per pair: more units than the 2 CTAs per SM
    idx = torch.arange(B) % distinct
    big = (feats[idx].cuda(), ki[idx], kj[idx], [ts[i] for i in idx.tolist()], size)
    a = run(mv, *big)
    assert_same_bits(a, run(mv, *big))
    for b in range(distinct):
        alone = run(mv, feats[b:b + 1].cuda(), ki[b:b + 1], kj[b:b + 1], [ts[b]], size)
        for x, y in zip(alone[:4], a[:4]):
            xb = x.view(torch.int32) if x.dtype == torch.float32 else x
            yb = y.view(torch.int32) if y.dtype == torch.float32 else y
            assert torch.equal(xb[0], yb[b])


def test_graph_capture(mv, syn):
    feats, ki, kj, ts, size = batch(syn, 3500, 4, C=128, h=50, w=50, K=30, image_size=800)
    feats2, ki2, kj2, _, _ = batch(syn, 3600, 4, C=128, h=50, w=50, K=30, image_size=800)
    f, a, b = feats.cuda(), ki.cuda(), kj.cuda()
    t = torch.tensor(ts, dtype=torch.float32, device="cuda")
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")
    mv.spair.compute_errors_batch(f, a, b, t, size, hits=hits)  # warm-up: shared-memory opt-in, allocator
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        hits.zero_()
        with torch.cuda.graph(g, stream=s):
            out = mv.spair.compute_errors_batch(f, a, b, t, size, hits=hits)
    torch.cuda.current_stream().wait_stream(s)
    f.copy_(feats2.cuda())
    a.copy_(ki2.cuda())
    b.copy_(kj2.cuda())
    hits.zero_()
    g.replay()
    torch.cuda.synchronize()
    got = tuple(x.cpu() for x in out) + (hits.cpu(),)
    h2 = torch.zeros(2, dtype=torch.int64, device="cuda")
    want = tuple(x.cpu() for x in mv.spair.compute_errors_batch(feats2.cuda(), ki2, kj2, t, size, hits=h2)) + (h2.cpu(),)
    assert_same_bits(got, want)


def test_agrees_with_first_form(mv, syn):
    """the timed size (768 x 50 x 50, K = 30, 16 pairs): the tiled and the first form pick the same pixel wherever the
    oracle's gap separates them; errors and counts agree."""
    feats, ki, kj, ts, size = batch(syn, 3700, 16, C=768, h=50, w=50, K=30, image_size=800)
    new = run(mv, feats.cuda(), ki, kj, ts, size)
    old = first_form(mv, feats, ki, kj, ts, size)
    same = new[3] == old[3]
    assert same.float().mean() >= 0.99
    for b in range(feats.shape[0]):
        _, _, oisame, _, heat = restated.spair_compute_errors(feats[b], ki[b], kj[b], ts[b], size, return_pred=True)
        flat = heat.flatten(1)
        top2 = torch.topk(flat, 2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-5
        assert torch.equal(new[3][b][clear], old[3][b][clear])
        assert torch.equal(new[0][b] >= 0, old[0][b] >= 0)
        m = same[b] & (new[0][b] >= 0)
        torch.testing.assert_close(new[0][b][m], old[0][b][m], rtol=0, atol=1e-5)
    assert new[4][0] == old[4][0] and abs(int(new[4][1]) - int(old[4][1])) <= int((~same).sum())


def test_no_candidate_gives_pixel_zero(mv, syn):
    """an all-NaN image j: no pixel is a candidate, pred is 0 as in the first form."""
    feats, ki, kj, ts, size = batch(syn, 3800, 3, C=64, h=20, w=20, K=20, image_size=320)
    feats[1, 1] = float("nan")
    new = run(mv, feats.cuda(), ki, kj, ts, size)
    old = first_form(mv, feats, ki, kj, ts, size)
    assert bool((new[3][1] == 0).all()) and bool((old[3][1] == 0).all())
    assert torch.equal(new[0][1] >= 0, old[0][1] >= 0)


def test_routes(mv, syn, monkeypatch):
    """maps above 256 pixels call the tiled entry point once with their MV_FEAT_* value and a workspace."""
    L = mv._lib
    feats, ki, kj, ts, size = batch(syn, 3900, 2, C=48, h=20, w=20, K=8, image_size=320)
    calls = []
    real = L.call
    monkeypatch.setattr(L, "call", lambda name, *a: (calls.append((name, a[1])), real(name, *a))[1])
    mv.spair.compute_errors_batch(feats.cuda(), ki, kj, ts, size)
    mv.spair.compute_errors_batch(feats.to(torch.bfloat16).cuda(), ki, kj, ts, size)
    assert calls == [("mv_spair_match_batch_tiled", L.MV_FEAT_F32), ("mv_spair_match_batch_tiled", L.MV_FEAT_BF16)]


def test_vit_b16_features_at_800(mv, syn):
    """random-init ViT-B/16 maps at the reference's 800-pixel input (768 x 50 x 50) through the tiled form, fp32 and bf16."""
    bb = importlib.import_module("midvision-probe_b200.backbones")
    model = bb.DenseViT(bb.vit_b16(0, img_size=800), multilayer=False).cuda()
    maps, kps = [], []
    with torch.no_grad():
        for s in range(3):
            maps.append(model.features(bb._pair_images(2000 + s, 800, 800, True, 0.5).cuda()))
            kps.append(syn.spair_pair(s, C=8, h=50, w=50, K=30, image_size=800))
    feats = torch.stack(maps).float()
    assert feats.shape[1:] == (2, 768, 50, 50)
    ki, kj = torch.stack([p["kps_i"] for p in kps]), torch.stack([p["kps_j"] for p in kps])
    ts = [p["thresh_scale"] for p in kps]
    check_oracle(mv, feats.cpu(), ki, kj, ts, 800)
    f16 = feats.to(torch.bfloat16)
    assert_same_bits(run(mv, f16, ki, kj, ts, 800), run(mv, f16.float(), ki, kj, ts, 800))
