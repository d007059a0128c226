"""SPair batches at the reference's 800-pixel input: the tiled form (mv_spair_match_batch_tiled, what compute_errors_batch
takes for maps above 256 pixels) against the first form (one CTA per pair, mv_spair_match_batch / _typed).

    python tools/spair_large_probe.py [--quick] > profiles/r3_spair_large_probe.jsonl

Shapes: 768 x 50 x 50, K = 30 (ViT-B/16 at 800 px); 768 x 57 x 57, K = 30 (ViT/14); 768 x 28 x 28, K = 20; 2048 x 25 x 25,
K = 30 (stride-32 CNN).  B in {16, 64, 256}.  16 distinct synthetic pairs cycled, materialised on the device; a shape's
batch is copied as often as needed to pass 300 MB and the copies are used in turn, so that every launch reads its maps from
HBM, not from the 126 MB L2.  Arms, alternated round by round (CUDA events, each warmed up):
  first_fp32 / first_bf16   the first form (mv_spair_match_batch / mv_spair_match_batch_typed)
  tiled_fp32 / tiled_bf16   spair.compute_errors_batch: the tiled form, its workspace allocated per call
Bytes model per pair: image j once (C * h*w * element size) plus the distinct 32-byte sectors of image i that the 4K
key-point taps touch.  One JSON line per (shape, B, arm): ms per launch, pairs/s, modelled bytes over the time and that rate
over the device-to-device copy peak measured in the same run, the speed-up of the tiled form over the first form of the same
element type, the card's name and power limit.  Before timing, at every timed size: the tiled bf16 outputs are asserted
bit-identical to the tiled fp32 outputs of the widened map, and the tiled and first forms' arg-max agreement is recorded
(`pred_agree`, with PCK counts of both).
"""
import importlib
import json
import math
import os
import sys
from ctypes import c_float

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
mv = importlib.import_module("midvision-probe_b200")
syn = importlib.import_module("midvision-probe_b200.synthetic")
from spair16_probe import card, copy_peak, timed  # noqa: E402

L = mv._lib
SHAPES = [(768, 50, 50, 30), (768, 57, 57, 30), (768, 28, 28, 20), (2048, 25, 25, 30)]
BATCHES = [16, 64, 256]
SIZE = 800
DISTINCT = 16


def sectors_i(ki, C, h, w, elem):
    """distinct 32-byte sectors of image i that the bilinear taps of the key points read (per pair, summed)."""
    total = 0
    for k in ki:
        ix = ((k[:, 0] / SIZE * 2 - 1 + 1) / 2) * (w - 1)
        iy = ((k[:, 1] / SIZE * 2 - 1 + 1) / 2) * (h - 1)
        x0, y0 = ix.floor().long(), iy.floor().long()
        taps = torch.cat([(y0 + dy).clamp(0, h - 1) * w + (x0 + dx).clamp(0, w - 1) for dy in (0, 1) for dx in (0, 1)]).unique()
        sec = ((torch.arange(C)[:, None] * h * w + taps[None, :]) * elem // 32).unique()
        total += sec.numel()
    return total


def first_form(feats, dtype, ki, kj, ts, out, hits):
    B, _, C, h, w = feats.shape
    K = ki.shape[1]
    args = (B, C, h, w, L.ptr(ki), L.ptr(kj), K, ki.shape[2], L.ptr(ts), c_float(float(SIZE)), c_float(0.10), L.ptr(out[3]),
            L.ptr(out[0]), L.ptr(out[1]), L.ptr(out[2]), L.ptr(hits), None, 0, mv.correspondence._stream())
    if dtype == torch.float32:
        L.call("mv_spair_match_batch", L.ptr(feats), *args)
    else:
        L.call("mv_spair_match_batch_typed", L.ptr(feats), L.MV_FEAT_BF16, *args)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("spair_large_probe: needs a CUDA device")
    quick = "--quick" in sys.argv
    peak = copy_peak(2 if quick else 5)
    gpu, power = card()
    for C, h, w, K in SHAPES:
        pairs = [syn.spair_pair(9000 + i, C=C, h=h, w=w, K=K, image_size=SIZE) for i in range(DISTINCT)]
        base = torch.stack([p["feats"] for p in pairs]).cuda()
        ki0 = torch.stack([p["kps_i"] for p in pairs])
        kj0 = torch.stack([p["kps_j"] for p in pairs])
        ts0 = torch.tensor([p["thresh_scale"] for p in pairs], dtype=torch.float32)
        sec = {e: sectors_i(ki0, C, h, w, e) / DISTINCT for e in (4, 2)}
        for B in BATCHES:
            idx = torch.arange(B) % DISTINCT
            ki, kj, ts = ki0[idx].cuda(), kj0[idx].cuda(), ts0[idx].cuda()
            f32 = base[idx.cuda()].contiguous()
            copies = max(1, math.ceil(300e6 / f32.numel() / 4))
            maps = {torch.float32: [f32] + [f32.clone() for _ in range(copies - 1)]}
            maps[torch.bfloat16] = [m.to(torch.bfloat16) for m in maps[torch.float32]]
            turn = {"i": 0}
            hits = torch.zeros(2, dtype=torch.int64, device="cuda")
            out = (torch.empty((B, K), device="cuda"), torch.empty((B, K), device="cuda"),
                   torch.empty((B, K), dtype=torch.int32, device="cuda"), torch.empty((B, K), dtype=torch.int32, device="cuda"))

            def pick(dt):
                turn["i"] += 1
                return maps[dt][turn["i"] % copies]

            variants = {
                "first_fp32": lambda: first_form(pick(torch.float32), torch.float32, ki, kj, ts, out, hits),
                "tiled_fp32": lambda: mv.spair.compute_errors_batch(pick(torch.float32), ki, kj, ts, SIZE, hits=hits),
                "first_bf16": lambda: first_form(pick(torch.bfloat16), torch.bfloat16, ki, kj, ts, out, hits),
                "tiled_bf16": lambda: mv.spair.compute_errors_batch(pick(torch.bfloat16), ki, kj, ts, SIZE, hits=hits),
            }
            # outputs at the timed size: tiled bf16 == tiled fp32 on the widened map (bits); tiled against first form
            bf, wid = maps[torch.bfloat16][0], maps[torch.bfloat16][0].float()
            ht, hw_, hf = (torch.zeros(2, dtype=torch.int64, device="cuda") for _ in range(3))
            a = mv.spair.compute_errors_batch(bf, ki, kj, ts, SIZE, hits=ht)
            b = mv.spair.compute_errors_batch(wid, ki, kj, ts, SIZE, hits=hw_)
            for x, y in zip(a, b):
                x = x.view(torch.int32) if x.dtype == torch.float32 else x
                y = y.view(torch.int32) if y.dtype == torch.float32 else y
                assert torch.equal(x, y), "tiled bf16 and tiled fp32 on the widened map disagree"
            assert torch.equal(ht, hw_)
            del wid
            t32 = mv.spair.compute_errors_batch(f32, ki, kj, ts, SIZE, hits=ht.zero_())
            first_form(f32, torch.float32, ki, kj, ts, out, hf)
            agree = float((t32[3] == out[3]).float().mean())
            pck = (ht.tolist(), hf.tolist())
            del a, b, t32

            for fn in variants.values():
                fn()
                fn()
            torch.cuda.synchronize()
            ms = timed(variants, 2 if quick else 5, 2 if quick else 5)
            for name, t in ms.items():
                elem = 4 if name.endswith("fp32") else 2
                byts = B * (C * h * w * elem + 32 * sec[elem])
                gbs = byts / (t * 1e-3) / 1e9
                other = ("first_" if name.startswith("tiled") else "tiled_") + name.split("_")[1]
                print(json.dumps({
                    "arm": name, "pairs": B, "C": C, "h": h, "w": w, "K": K, "gpu": gpu, "power_limit": power,
                    "ms_per_launch": round(t, 4), "pairs_per_s": round(B / (t * 1e-3)), "model_bytes": int(byts),
                    "model_gbs": round(gbs, 1), "copy_peak_gbs": round(peak, 1), "share_of_copy_peak": round(gbs / peak, 3),
                    "tiled_speedup": round((ms[other] / t) if name.startswith("tiled") else (t / ms[other]), 2),
                    "pred_agree": round(agree, 5), "hits_tiled_first": pck, "bf16_equals_widened_fp32": True,
                }), flush=True)
            del maps, f32, variants
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
