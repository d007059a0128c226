"""SPair batches on 16-bit feature maps: the bf16 / fp16 streaming kernel against the route 16-bit maps took before (torch
widening to fp32 + the fp32 kernel), at the benchmark's SPair shape.

    python tools/spair16_probe.py [--quick] > profiles/r3_spair_16bit_probe.jsonl

2368 pairs per launch (bench.py's SPAIR_BATCH: 8 per CTA at 2 CTAs x 148 SMs), C = 768, 14 x 14, K = 20; 32 distinct
synthetic pairs cycled, materialised on the device: 2.85 GB of fp32 / 1.43 GB of 16-bit features per launch, larger than
the 126 MB L2.  The arms are alternated round by round (CUDA events, every arm warmed up):
  fp32           fp32 features through mv_spair_match_batch
  bf16_widen     bf16 features the way compute_errors_batch took them before: .float() (a torch copy) + the fp32 kernel,
                 the widening timed with the launch
  bf16           bf16 features through mv_spair_match_batch_typed (the 16-bit streaming kernel)
  f16            fp16 likewise
  bf16_tf32      bf16 with spair.set_heatmap_precision("tf32")
One JSON line per arm: ms per launch, pairs/s, algorithmic bytes (B * 2 * C * h * w * element size: the map read once)
over the time, and that rate over the device-to-device copy peak measured in the same run (read + write bytes of a 2 GiB
torch copy, CUDA events; bench.py's peaks() figure is recorded beside it), with the card's name and power limit.  The
outputs of bf16_widen and bf16 are asserted bit-identical at the timed size before anything is printed.
"""
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
mv = importlib.import_module("midvision-probe_b200")
syn = importlib.import_module("midvision-probe_b200.synthetic")
sp = mv.spair

B, C, H, W, K = 2368, 768, 14, 14, 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
        name, power = [x.strip() for x in out.split(",")]
    except Exception as e:  # the figure is still labelled with what torch reports
        name, power = torch.cuda.get_device_name(), f"unknown ({type(e).__name__})"
    return name, power


def bench_peak():
    """bench.py's peaks(): MEASURED_PEAKS.json's hbm_gbs where that file exists, else its fallback figure."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


def copy_peak(rounds):
    """device-to-device copy rate: (read + write bytes) / time of a 2 GiB torch copy, best of `rounds`."""
    n = 1 << 29
    src, dst = torch.ones(n, device="cuda"), torch.empty(n, device="cuda")
    for _ in range(3):
        dst.copy_(src)
    best = None
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            dst.copy_(src)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 5
        best = ms if best is None else min(best, ms)
    del src, dst
    return 2 * 4 * n / (best * 1e-3) / 1e9


def timed(variants, iters, rounds):
    """variants: name -> callable; alternated round by round; returns ms per call"""
    ev = {k: [] for k in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            ev[name].append((a, b))
    torch.cuda.synchronize()
    return {k: sum(a.elapsed_time(b) for a, b in v) / (len(v) * iters) for k, v in ev.items()}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("spair16_probe: needs a CUDA device")
    quick = "--quick" in sys.argv
    pairs = [syn.spair_pair(i, C=C, h=H, w=W, K=K) for i in range(32)]
    idx = torch.arange(B) % 32
    f32 = torch.stack([p["feats"] for p in pairs]).cuda()[idx.cuda()].contiguous()
    bf16, f16 = f32.to(torch.bfloat16), f32.to(torch.float16)
    ki = torch.stack([p["kps_i"] for p in pairs])[idx].cuda()
    kj = torch.stack([p["kps_j"] for p in pairs])[idx].cuda()
    ts = torch.tensor([p["thresh_scale"] for p in pairs], dtype=torch.float32)[idx].cuda()
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")

    def call(feats):
        return lambda: sp.compute_errors_batch(feats, ki, kj, ts, 224, hits=hits)

    def tf32(feats):
        def fn():
            prev = sp.set_heatmap_precision("tf32")
            try:
                sp.compute_errors_batch(feats, ki, kj, ts, 224, hits=hits)
            finally:
                sp.set_heatmap_precision(prev)
        return fn

    variants = {"fp32": call(f32), "bf16_widen": lambda: sp.compute_errors_batch(bf16.float(), ki, kj, ts, 224, hits=hits),
                "bf16": call(bf16), "f16": call(f16), "bf16_tf32": tf32(bf16)}
    elem = {"fp32": 4, "bf16_widen": 2, "bf16": 2, "f16": 2, "bf16_tf32": 2}

    # the new route against the old one at the timed size: every output, the PCK counts and the confusion matrix
    outs = []
    for feats in (bf16.float(), bf16):
        h = torch.zeros(2, dtype=torch.int64, device="cuda")
        conf = torch.zeros((K, K), dtype=torch.int64, device="cuda")
        outs.append(tuple(sp.compute_errors_batch(feats, ki, kj, ts, 224, hits=h, confusion=conf)) + (h, conf))
    for x, y in zip(*outs):
        x = x.view(torch.int32) if x.dtype == torch.float32 else x
        y = y.view(torch.int32) if y.dtype == torch.float32 else y
        assert torch.equal(x, y), "bf16 kernel and widened fp32 kernel disagree"
    del outs

    for fn in variants.values():
        fn()
        fn()
    torch.cuda.synchronize()
    ms = timed(variants, 2 if quick else 10, 2 if quick else 6)
    peak = copy_peak(2 if quick else 5)
    bpeak, bkind = bench_peak()
    gpu, power = card()
    for name, t in ms.items():
        byts = B * 2 * C * H * W * elem[name]
        gbs = byts / (t * 1e-3) / 1e9
        print(json.dumps({
            "arm": name, "pairs": B, "C": C, "h": H, "w": W, "K": K, "gpu": gpu, "power_limit": power,
            "ms_per_launch": round(t, 4), "pairs_per_s": round(B / (t * 1e-3)), "algorithmic_bytes": byts,
            "algorithmic_gbs": round(gbs, 1), "copy_peak_gbs": round(peak, 1), "share_of_copy_peak": round(gbs / peak, 3),
            "bench_peak_gbs": bpeak, "bench_peak_kind": bkind, "vs_bf16_widen": round(ms["bf16_widen"] / t, 3),
            "bf16_equals_widened_fp32": True,
        }), flush=True)


if __name__ == "__main__":
    main()
