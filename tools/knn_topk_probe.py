"""k > 2 nearest neighbours: kernel 2's row top-KP epilogue + fp32 re-rank against the blocked fp32 search it replaces.

    python tools/knn_topk_probe.py [--quick] > profiles/r3_knn_topk_probe.jsonl

One JSON line per shape (NAVI-shaped 5024^2 x 3072 cosine k = 5 and 8, ScanNet-shaped 18231^2 x 2048 cosine k = 8,
19200^2 x 768 L2 k = 8), each with the card's name and power limit read in the same run.  CUDA events, every shape
warmed up, the variants alternated round by round; inputs stay in device memory (not flushed from L2 between launches):
  topk_ms     mv_k2_sim_topk_ld: the GEMM kernel with the top-KP epilogue + its row-merge launch; TFLOP/s of 2 n m K
              (K = product columns, augmentation included) and the share of 1647.2 TFLOP/s (16-bit operands, the
              kernel-2 denominator of DESIGN.md section 4) or of half of it (tf32)
  top2_ms     mv_k2_sim_top2_ld on the same operands (GEMM kernel + column memset + row merge)
  rerank_ms   mv_knn_rerank
  public_ms   the whole public call (knn_points cosine / faiss_knn), operand preparation included
  blocked_ms  the blocked fp32 search the public call took before (normalise, torch GEMM + top-k per 4096 rows, gather)
  agree       fraction of (row, position) entries where the fused and blocked indices agree; agree_gap the same on the
              positions separated from both neighbours by > 1e-3 (cosine: similarity; L2: relative squared distance)
"""
import importlib
import json
import os
import subprocess
import sys
from ctypes import c_size_t

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
mv = importlib.import_module("midvision-probe_b200")
C_ = mv.correspondence
L = mv._lib

PEAK_16BIT = 1647.2  # TFLOP/s, DESIGN.md section 4


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
        name, power = [x.strip() for x in out.split(",")]
    except Exception as e:  # the figure is still labelled with what torch reports
        name, power = torch.cuda.get_device_name(), f"unknown ({type(e).__name__})"
    return name, power


def blocked_knn(X, Y, k, metric):
    """the k > 2 route the public functions took before: exact blocked fp32 search (+ the cosine distances)"""
    if metric == "l2":
        return C_._exact_knn_blocks(X, Y, k)
    Xn, Yn = F.normalize(X, dim=-1), F.normalize(Y, dim=-1)
    _, idx = C_._exact_knn_blocks(Xn, Yn, k)
    return 1 - F.cosine_similarity(Yn[idx], Xn[:, None, :], dim=-1), idx


def timed(variants, iters, rounds):
    """variants: name -> callable; alternated round by round; returns ms per call"""
    ev = {k: [] for k in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters[name]):
                fn()
            b.record()
            ev[name].append((a, b, iters[name]))
    torch.cuda.synchronize()
    return {k: sum(a.elapsed_time(b) for a, b, _ in v) / sum(n for _, _, n in v) for k, v in ev.items()}


def shape_line(name, n, m, C, k, metric, quick):
    g = torch.Generator(device="cuda").manual_seed(n + m + C + k)
    X = torch.randn(n, C, device="cuda", generator=g)
    Y = torch.randn(m, C, device="cuda", generator=g)
    kp = 8 if k <= 6 else 16
    st = C_._stream()
    if metric == "cosine":
        (A16, A32), (B16, B32), _ = C_._rows_pair(X, Y, X.device)
        A, B, Ck, dtype = C_._k2_operands(A16, A32, B16, B32, C)
        Q, T, rr_metric = A32, B32, L.MV_METRIC_COSINE
        public = lambda: C_.knn_points(X, Y, k, "cosine")  # noqa: E731
    else:
        A, B = C_._l2_operands(X, Y)
        Ck, dtype = A.shape[1], L.MV_DTYPE_TF32
        Q, T, rr_metric = X, Y, L.MV_METRIC_L2SQ
        public = lambda: C_.faiss_knn(X, Y, k)  # noqa: E731
    lib = L.load()
    cl = C_._CFG["cluster"]
    rv, ri = torch.empty((n, kp), device="cuda"), torch.empty((n, kp), dtype=torch.int32, device="cuda")
    wsk = lib.mv_k2_topk_workspace_bytes(n, m, kp)
    ws_k = torch.empty(wsk, dtype=torch.uint8, device="cuda")
    rv2, ri2 = torch.empty((n, 2), device="cuda"), torch.empty((n, 2), dtype=torch.int32, device="cuda")
    cb = torch.empty(m, dtype=torch.int64, device="cuda")
    ws2 = lib.mv_k2_workspace_bytes(n, m)
    ws_2 = torch.empty(ws2, dtype=torch.uint8, device="cuda")
    dd, di = torch.empty((n, k), device="cuda"), torch.empty((n, k), dtype=torch.int32, device="cuda")

    def topk():
        L.call("mv_k2_sim_topk_ld", L.ptr(A), A.shape[1], L.ptr(B), B.shape[1], n, m, Ck, None, None, dtype, cl, kp, L.ptr(rv),
               L.ptr(ri), L.ptr(ws_k), c_size_t(wsk), st)

    def top2():
        L.call("mv_k2_sim_top2_ld", L.ptr(A), A.shape[1], L.ptr(B), B.shape[1], n, m, Ck, None, None, dtype, cl, L.ptr(rv2),
               L.ptr(ri2), L.ptr(cb), L.ptr(ws_2), c_size_t(ws2), st)

    def rerank():
        L.call("mv_knn_rerank", L.ptr(Q), Q.stride(0), L.ptr(T), T.stride(0), Q.shape[1], None, n, L.ptr(ri), kp, k, rr_metric,
               L.ptr(dd), L.ptr(di), st)

    blocked = lambda: blocked_knn(X, Y, k, metric)  # noqa: E731
    variants = {"topk": topk, "top2": top2, "rerank": rerank, "public": public, "blocked": blocked}
    for fn in variants.values():  # warm-up: module loads, function attributes, cuBLAS algorithm choice
        fn()
        fn()
    torch.cuda.synchronize()
    iters = {"topk": 20, "top2": 20, "rerank": 20, "public": 10, "blocked": 2}
    if quick:
        iters = {key: 1 for key in iters}
    ms = timed(variants, iters, 2 if quick else 5)

    # old and new outputs on the timed inputs
    d_new, i_new = public()
    d_old, i_old = blocked_knn(X, Y, k + 1, metric)
    i_new, i_old = i_new.cpu(), i_old.cpu()
    od = d_old.double().cpu()
    clear = torch.ones((n, k), dtype=torch.bool)
    rel = (lambda x: 1e-3 * x) if metric == "l2" else (lambda x: 1e-3)
    for j in range(k):
        if j > 0:
            clear[:, j] &= od[:, j] - od[:, j - 1] > rel(od[:, j - 1])
        clear[:, j] &= od[:, j + 1] - od[:, j] > rel(od[:, j])
    same = i_new == i_old[:, :k]
    flop = 2.0 * n * m * Ck
    peak = PEAK_16BIT if dtype != L.MV_DTYPE_TF32 else PEAK_16BIT / 2
    tflops = flop / (ms["topk"] * 1e-3) / 1e12
    gpu, power = card()
    return {
        "shape": name, "n": n, "m": m, "C": C, "k": k, "kp": kp, "metric": metric,
        "operands": {L.MV_DTYPE_BF16: "bf16", L.MV_DTYPE_F16: "f16c", L.MV_DTYPE_TF32: "tf32"}[dtype], "product_columns": Ck,
        "gpu": gpu, "power_limit": power,
        "topk_ms": round(ms["topk"], 4), "topk_tflops": round(tflops, 1), "topk_share_of_peak": round(tflops / peak, 3),
        "peak_tflops": peak, "top2_ms": round(ms["top2"], 4), "topk_over_top2": round(ms["topk"] / ms["top2"], 3),
        "rerank_ms": round(ms["rerank"], 4), "public_ms": round(ms["public"], 4), "blocked_ms": round(ms["blocked"], 4),
        "blocked_over_public": round(ms["blocked"] / ms["public"], 2),
        "agree": round(float(same.float().mean()), 5), "gap_fraction": round(float(clear.float().mean()), 4),
        "agree_gap": float(same[clear].float().mean()) if clear.any() else None,
    }


SHAPES = [
    ("navi_5024x5024x3072", 5024, 5024, 3072, 5, "cosine"),
    ("navi_5024x5024x3072", 5024, 5024, 3072, 8, "cosine"),
    ("scannet_18231x18231x2048", 18231, 18231, 2048, 8, "cosine"),
    ("stress_19200x19200x768", 19200, 19200, 768, 8, "l2"),
]


def main():
    if not torch.cuda.is_available():
        raise SystemExit("knn_topk_probe: needs a CUDA device")
    quick = "--quick" in sys.argv
    for name, n, m, C, k, metric in SHAPES:
        if quick:
            n, m = n // 8, m // 8
        print(json.dumps(shape_line(name, n, m, C, k, metric, quick)), flush=True)


if __name__ == "__main__":
    main()
