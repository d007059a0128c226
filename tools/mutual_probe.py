"""Mutual matching from one similarity product: kernel 2's column top-2 variant against the top-2 kernel, and the whole
mutual call against the two-product route it replaces.

    python tools/mutual_probe.py [--quick] [--out profiles/r3_mutual_probe.jsonl]

One JSON line per shape, each with the card's name and power limit read in the same run.  CUDA events around every call,
every arm warmed up first, the arms alternated call by call, and each call reads the next of several input sets, as many
as it takes for their operands to exceed 256 MB -- twice the 126 MB L2 -- so that no call finds its operands in L2:
  cols_ms    mv_k2_sim_top2_cols_ld (GEMM kernel with the row and column top-2 epilogue + row merge + column merge)
  top2_ms    mv_k2_sim_top2_ld on the same operands (GEMM kernel + column memset + row merge)
  TFLOP/s    2 n m K over the time, K = product columns (augmentation included)
  mutual_ms  get_mutual_correspondences on device-resident features (rows, one product, both kernel-3 passes, selection)
  bidir_ms   get_correspondences_ratio_test(bidirectional=True) on the same features: rows and a product per direction
"""
import importlib
import json
import os
import subprocess
import sys
from ctypes import c_size_t

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
mv = importlib.import_module("midvision-probe_b200")
C_ = mv.correspondence
L = mv._lib

ROTATE_BYTES = 256 << 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
        name, power = [x.strip() for x in out.split(",")]
    except Exception as e:  # the figure is still labelled with what torch reports
        name, power = torch.cuda.get_device_name(), f"unknown ({type(e).__name__})"
    return name, power


def timed(arms, calls):
    """arms: name -> list of callables (one per input set); alternated call by call; returns median ms per call"""
    ev = {k: [] for k in arms}
    for c in range(calls):
        for name, fns in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fns[c % len(fns)]()
            b.record()
            ev[name].append((a, b))
    torch.cuda.synchronize()
    return {k: sorted(a.elapsed_time(b) for a, b in v)[len(v) // 2] for k, v in ev.items()}


def sets_for(bytes_per_set):
    return max(2, min(16, -(-ROTATE_BYTES // bytes_per_set)))


def kernel_arms(n, m, Ck, pitch, dtype, nsets):
    """the two kernel-2 entry points on nsets random operand sets of (n, pitch) / (m, pitch) over Ck columns"""
    t = {L.MV_DTYPE_BF16: torch.bfloat16, L.MV_DTYPE_F16: torch.float16, L.MV_DTYPE_TF32: torch.float32}[dtype]
    lib = L.load()
    st = C_._stream()
    cl = C_._CFG["cluster"]
    rv, ri = torch.empty((n, 2), device="cuda"), torch.empty((n, 2), dtype=torch.int32, device="cuda")
    cv, ci = torch.empty((m, 2), device="cuda"), torch.empty((m, 2), dtype=torch.int32, device="cuda")
    cb = torch.empty(m, dtype=torch.int64, device="cuda")
    wc, w2 = lib.mv_k2_cols_workspace_bytes(n, m), lib.mv_k2_workspace_bytes(n, m)
    ws_c, ws_2 = torch.empty(wc, dtype=torch.uint8, device="cuda"), torch.empty(w2, dtype=torch.uint8, device="cuda")
    cols, top2 = [], []
    for s in range(nsets):
        g = torch.Generator(device="cuda").manual_seed(s)
        A = (torch.randn(n, pitch, device="cuda", generator=g) / pitch ** 0.5).to(t)
        B = (torch.randn(m, pitch, device="cuda", generator=g) / pitch ** 0.5).to(t)
        cols.append(lambda A=A, B=B: L.call("mv_k2_sim_top2_cols_ld", L.ptr(A), pitch, L.ptr(B), pitch, n, m, Ck, None, None, dtype,
                                            cl, L.ptr(rv), L.ptr(ri), L.ptr(cv), L.ptr(ci), L.ptr(cb), L.ptr(ws_c), c_size_t(wc), st))
        top2.append(lambda A=A, B=B: L.call("mv_k2_sim_top2_ld", L.ptr(A), pitch, L.ptr(B), pitch, n, m, Ck, None, None, dtype, cl,
                                            L.ptr(rv), L.ptr(ri), L.ptr(cb), L.ptr(ws_2), c_size_t(w2), st))
    return {"cols": cols, "top2": top2}


def public_arms(n, m, C, nsets):
    mutual, bidir = [], []
    for s in range(nsets):
        g = torch.Generator(device="cuda").manual_seed(100 + s)
        P1, P2 = torch.randn(n, C, device="cuda", generator=g), torch.randn(m, C, device="cuda", generator=g)
        mutual.append(lambda P1=P1, P2=P2: C_.get_mutual_correspondences(P1, P2, 1000))
        bidir.append(lambda P1=P1, P2=P2: C_.get_correspondences_ratio_test(P1, P2, 1000, bidirectional=True))
    return {"mutual": mutual, "bidir": bidir}


# name, n, m, product columns, operand pitch, operand type, features C of the whole-call arms (None: kernel only)
SHAPES = [
    ("navi_5024x5024x3080_f16c", 5024, 5024, 3080, 3136, L.MV_DTYPE_F16, 3072),
    ("scannet_lowrank_18231x18231x312_f16", 18231, 18231, 312, 320, L.MV_DTYPE_F16, None),
    ("scannet_18231x18231x2056_f16c", 18231, 18231, 2056, 2112, L.MV_DTYPE_F16, 2048),
    ("stress_19200x19200x768_bf16", 19200, 19200, 768, 768, L.MV_DTYPE_BF16, None),
]


def main():
    if not torch.cuda.is_available():
        raise SystemExit("mutual_probe: needs a CUDA device")
    quick = "--quick" in sys.argv
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join("profiles", "r3_mutual_probe.jsonl")
    gpu, power = card()
    lines = []
    for name, n, m, Ck, pitch, dtype, Cf in SHAPES:
        if quick:
            n, m = n // 8, m // 8
        esz = 4 if dtype == L.MV_DTYPE_TF32 else 2
        arms = kernel_arms(n, m, Ck, pitch, dtype, sets_for((n + m) * pitch * esz))
        if Cf is not None:
            arms.update(public_arms(n, m, Cf, sets_for((n + m) * Cf * 4)))
        for fns in arms.values():  # warm-up: module loads, function attributes, every input set once
            for fn in fns:
                fn()
        torch.cuda.synchronize()
        ms = timed(arms, 4 if quick else 40)
        flop = 2.0 * n * m * Ck
        rec = {"shape": name, "n": n, "m": m, "K": Ck, "operands": {L.MV_DTYPE_BF16: "bf16", L.MV_DTYPE_F16: "f16"}[dtype],
               "gpu": gpu, "power_limit": power, "input_sets": len(arms["cols"]),
               "cols_ms": round(ms["cols"], 4), "cols_tflops": round(flop / (ms["cols"] * 1e-3) / 1e12, 1),
               "top2_ms": round(ms["top2"], 4), "top2_tflops": round(flop / (ms["top2"] * 1e-3) / 1e12, 1),
               "cols_over_top2": round(ms["cols"] / ms["top2"], 3)}
        if Cf is not None:
            rec.update({"features_C": Cf, "mutual_ms": round(ms["mutual"], 4), "bidir_ms": round(ms["bidir"], 4),
                        "mutual_over_bidir": round(ms["mutual"] / ms["bidir"], 3)})
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if not quick:
        with open(out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
