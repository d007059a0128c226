"""SPair batches on bf16 / fp16 feature maps (mv_spair_match_batch_typed).  Widening a 16-bit value to fp32 is exact and the
16-bit kernels keep the fp32 kernels' channel chunks and summation order, so compute_errors_batch(f16) must equal
compute_errors_batch(f16.float()) BIT FOR BIT: pred, error_same, error_nn, index_nn, the PCK counts and the confusion
matrix.  Covered: the SPair shape, every key-point tile edge, a tail channel chunk, odd and even h*w, the first form
(h*w > 256, C % 8 != 0, a map that is not 16-byte aligned), more pairs than resident CTAs, both heat-map precisions,
host-resident input, the oracle, and ViT-B/16 features produced under bf16 autocast."""
import importlib

import pytest
import torch

from oracle import restated

pytestmark = pytest.mark.gpu

DTYPES = [torch.bfloat16, torch.float16]


def batch(syn, seed, B, C=768, h=14, w=14, K=20, image_size=224):
    pairs = [syn.spair_pair(seed + i, C=C, h=h, w=w, K=K, image_size=image_size) for i in range(B)]
    return (torch.stack([p["feats"] for p in pairs]), torch.stack([p["kps_i"] for p in pairs]),
            torch.stack([p["kps_j"] for p in pairs]), [p["thresh_scale"] for p in pairs], image_size)


def run(mv, feats, ki, kj, ts, image_size, kp_max=64):
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")
    conf = torch.zeros((kp_max, kp_max), dtype=torch.int64, device="cuda")
    out = mv.spair.compute_errors_batch(feats, ki, kj, ts, image_size, hits=hits, confusion=conf)
    return tuple(x.cpu() for x in out) + (hits.cpu(), conf.cpu())


def assert_bit_identical(mv, f16, ki, kj, ts, image_size, widened=None):
    """the 16-bit batch against the same batch widened to fp32 (or `widened`: an fp32 copy laid out like f16)."""
    a = run(mv, f16, ki, kj, ts, image_size)
    b = run(mv, f16.float() if widened is None else widened, ki, kj, ts, image_size)
    names = ("error_same", "error_nn", "index_nn", "pred", "hits", "confusion")
    for name, x, y in zip(names, a, b):
        assert x.dtype == y.dtype and x.shape == y.shape, name
        # bit patterns, not values: -0 == +0 but a sign flip would still show here
        xb = x.view(torch.int32) if x.dtype == torch.float32 else x
        yb = y.view(torch.int32) if y.dtype == torch.float32 else y
        assert torch.equal(xb, yb), f"{name} differs at {int((xb != yb).sum())} positions"
    assert int(a[4][0]) > 0  # key points in both images were scored
    return a


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
def test_spair_shape(mv, syn, dtype, precision):
    """the SPair shape (C = 768, 14 x 14, K = 20) in both heat-map precisions."""
    feats, ki, kj, ts, size = batch(syn, 300, 9)
    prev = mv.spair.set_heatmap_precision(precision)
    try:
        assert_bit_identical(mv, feats.to(dtype).cuda(), ki, kj, ts, size)
    finally:
        mv.spair.set_heatmap_precision(prev)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("K", [1, 8, 9, 20, 21, 25, 33, 64])
def test_keypoint_tile_edges(mv, syn, dtype, K):
    """every key-point tile size the launcher picks (KT = 8 .. 32) and its edges, including two tiles (K > 32)."""
    feats, ki, kj, ts, size = batch(syn, 400 + K, 4, C=48, K=K)
    assert_bit_identical(mv, feats.to(dtype).cuda(), ki, kj, ts, size)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("shape", [dict(C=72, h=16, w=16, K=40, image_size=256),   # 256 pixels, 24-channel tail chunk
                                   dict(C=104, h=15, w=15, K=17, image_size=240),  # odd h*w: 16-bit A loads, 8-channel tail
                                   dict(C=96, h=14, w=15, K=20, image_size=224)])  # even h*w, not square
def test_tail_chunks_and_pixel_counts(mv, syn, dtype, precision, shape):
    feats, ki, kj, ts, size = batch(syn, 500, 3, **shape)
    prev = mv.spair.set_heatmap_precision(precision)
    try:
        assert_bit_identical(mv, feats.to(dtype).cuda(), ki, kj, ts, size)
    finally:
        mv.spair.set_heatmap_precision(prev)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [dict(C=64, h=20, w=20, K=20, image_size=320),  # h*w > 256
                                   dict(C=44, h=14, w=14, K=20, image_size=224)])  # C % 8 != 0
def test_first_form(mv, syn, dtype, shape):
    feats, ki, kj, ts, size = batch(syn, 600, 3, **shape)
    assert_bit_identical(mv, feats.to(dtype).cuda(), ki, kj, ts, size)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("offset", [1, 2, 3, 4])
def test_misaligned_map_takes_the_first_form(mv, syn, dtype, offset):
    """a map 2-8 bytes past a 16-byte boundary runs the first form; the fp32 reference is laid out 4 bytes off as well,
    so that it runs the first form too (the streaming form sums in another order)."""
    feats, ki, kj, ts, size = batch(syn, 700 + offset, 3, C=64)
    n = feats.numel()

    def placed(dt, off):
        buf = torch.zeros(n + 8, dtype=dt, device="cuda")
        f = buf[off:off + n].view(feats.shape)
        f.copy_(feats.to(dtype).to(dt))
        return f

    f16 = placed(dtype, offset)
    f32 = placed(torch.float32, 1)
    assert f16.data_ptr() % 16 == 2 * offset and f32.data_ptr() % 16 == 4
    assert_bit_identical(mv, f16, ki, kj, ts, size, widened=f32)


@pytest.mark.parametrize("dtype", DTYPES)
def test_more_pairs_than_resident_ctas(mv, syn, dtype):
    shape = dict(C=48, h=14, w=14, K=20, image_size=224)
    distinct = 37
    feats, ki, kj, ts, size = batch(syn, 800, distinct, **shape)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    B = 4 * sm + 45
    idx = torch.arange(B) % distinct
    assert_bit_identical(mv, feats[idx].to(dtype).cuda(), ki[idx], kj[idx], [ts[i] for i in idx.tolist()], size)


@pytest.mark.parametrize("dtype", DTYPES)
def test_host_resident_input(mv, syn, dtype):
    """a 16-bit map on the host is uploaded as it is; the reference widens it on the host."""
    feats, ki, kj, ts, size = batch(syn, 900, 5)
    assert_bit_identical(mv, feats.to(dtype), ki, kj, ts, size)


def test_routes(mv, syn, monkeypatch):
    """16-bit maps call the typed entry point once with their MV_FEAT_* value; fp32 keeps its one mv_spair_match_batch call."""
    L = mv._lib
    feats, ki, kj, ts, size = batch(syn, 950, 2, C=48)
    calls = []
    real = L.call
    monkeypatch.setattr(L, "call", lambda name, *a: (calls.append((name, a[1] if name.endswith("_typed") else None)), real(name, *a))[1])
    mv.spair.compute_errors_batch(feats.cuda(), ki, kj, ts, size)
    mv.spair.compute_errors_batch(feats.to(torch.bfloat16).cuda(), ki, kj, ts, size)
    mv.spair.compute_errors_batch(feats.to(torch.float16), ki, kj, ts, size)
    assert calls == [("mv_spair_match_batch", None), ("mv_spair_match_batch_typed", L.MV_FEAT_BF16),
                     ("mv_spair_match_batch_typed", L.MV_FEAT_F16)]


@pytest.mark.parametrize("dtype", DTYPES)
def test_against_oracle(mv, syn, dtype):
    """the 16-bit batch against the fp64 oracle on the widened map: arg-max identical wherever the top-2 heat-map gap
    exceeds 1e-5, errors to 1e-5, the key points kept bit-exact."""
    feats, ki, kj, ts, size = batch(syn, 1000, 6)
    f16 = feats.to(dtype)
    es, en, inn, pred = (x.cpu() for x in mv.spair.compute_errors_batch(f16.cuda(), ki, kj, ts, size))
    for b in range(f16.shape[0]):
        oes, oen, oisame, oinn, heat = restated.spair_compute_errors(f16[b].float(), ki[b], kj[b], ts[b], size, return_pred=True)
        flat = heat.flatten(1)
        top2 = torch.topk(flat, 2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-5
        assert torch.equal(pred[b].long()[clear], flat.argmax(1)[clear])
        assert torch.equal((es[b] >= 0).nonzero().squeeze(1), oisame)
        ok = clear[oisame]
        torch.testing.assert_close(es[b][oisame][ok], oes[ok], rtol=0, atol=1e-5)


def test_vit_features_under_bf16_autocast(mv):
    """SPair-shaped pairs whose maps come out of a random-init ViT-B/16 run under bf16 autocast, kept in bf16."""
    bb = importlib.import_module("midvision-probe_b200.backbones")
    model = bb.DenseViT(bb.vit_b16(0, img_size=224), multilayer=False).cuda()
    pairs = [bb.spair_backbone_pair(s, model, device="cuda", noise=0.5) for s in range(6)]
    maps = []
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for s in range(6):
            maps.append(model.features(bb._pair_images(2000 + s, 224, 224, True, 0.5).cuda()).to(torch.bfloat16))
    feats = torch.stack(maps)
    assert feats.shape[1:] == (2, 768, 14, 14)
    assert_bit_identical(mv, feats, torch.stack([p["kps_i"] for p in pairs]), torch.stack([p["kps_j"] for p in pairs]),
                         [p["thresh_scale"] for p in pairs], 224)
