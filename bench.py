#!/usr/bin/env python
"""Benchmark of the dense-correspondence matching path (BASELINE.json metric: image pairs / s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload navi|scannet|spair|all]
                    [--pairs P] [--features backbone|gaussian] [--dtype f16|bf16|tf32] [--dump-outputs DIR]

One "step" = one batch of PAIRS_PER_STEP synthetic image pairs through the hot path (kernels 1-3 + scoring).
The HEADLINE workload (top-level keys of the one JSON line) is BASELINE.json configs[1]: NAVI-shaped pairs, ViT-B/16 @
448, 4-block concat 3072-d features on a 28 x 28 grid, 112 x 112 xyz grid, 1000 correspondences; pair i runs on
rank i mod N and the integer hit counts are all-reduced once over NCCL ("weak" scaling: every rank processes the
same number of pairs).  With the default --workload all the same line also carries, measured in the same process:

    workloads.scannet / workloads.spair   configs[2] / configs[0]: value, e2e, roofline, clocks each
    k1                                    kernel 1 alone (CUDA events): bytes, us, GB/s against the HBM copy peak
    k2_stress                             configs[4]: 19200 x 19200 x 768, bf16 / f16 / tf32, kernel 2 alone (N = 1)
    sharded_set                           configs[3] in small: a FIXED seeded set of pairs, pair i -> rank i mod N,
                                          the reduced hit vector and its SHA-1 (equal for every N); --pairs 10000 runs
                                          the full-size set as the headline with "scaling": "strong"
    backbone                              the random-init backbone forward next to the matching path

`value`        pairs/s with the feature maps / xyz grids resident in HBM (device-side loop, no host sync).
`e2e`          pairs/s through the reference-facing helper estimate_correspondence_xyz called with HOST tensors (pinned),
               H2D / D2H copies and the helper's own syncs inside the timed region; `e2e_pageable` = the same with plain
               pageable tensors, which is what the reference's callers hold (evaluate_navi_correspondence.py:149-150).
`roofline`     kernel 2 (the tcgen05 similarity GEMM) timed with CUDA events over the same steps.
`cpu_baseline` (rank 0, N = 1) the CPU oracle port of the reference on a bounded sample.
`--impl reference` times that CPU port alone with all host threads (the reference tree is Python that cannot travel to
the GPU box and needs faiss-gpu, which this image does not have).
"""
import argparse
import hashlib
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PAIRS_PER_STEP = 32
POOL = 16          # distinct pairs cycled through; their working set (~190 MB / pair) exceeds the 126 MB L2
NUM_CORR = 1000
THR = {"navi": ([0.01, 0.02, 0.05], [5, 25, 50]),                         # evaluate_navi_correspondence.py:200-212
       "scannet": ([0.01, 0.02, 0.05, 0.10], [5, 10, 20, 30, 40, 50])}    # render_scannet_correspondence.py:129-147, :253-264
METRIC = "image pairs/sec for dense mutual-NN matching"
SHARDED_PAIRS = 256  # size of the fixed set of the default run's sharded_set record
REF_WALL_CAP_S = 150.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nme, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


WORKLOAD_NAME = {
    "navi": "NAVI-shaped dense correspondence, ViT-B/16 @448 4-block concat (3072, 28, 28) -> 112x112 xyz grid, "
            "num_corr 1000 (BASELINE.json configs[1])",
    "scannet": "ScanNet-shaped, ResNet-50 layer4 (2048, 15, 20) -> 120x160 depth, 19200x19200 similarity, "
               "num_corr 1000 (BASELINE.json configs[2])",
    "spair": "SPair-shaped pairs: (2, 768, 14, 14) features, 20 key points, fused batched matching "
             "(BASELINE.json configs[0])"}
FEATURES_NAME = {
    "backbone": "random-init frozen backbone (ViT-B/16 blocks [2,5,8,11] concat / ResNet-50 layer4) on seeded smooth images, "
                "image 1 = image 0 + photometric change + noise",
    "gaussian": "seeded N(0,1) maps of the backbone's output shape"}


class Ctx:
    """process-wide state of one bench run."""

    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.mv = importlib.import_module("midvision-probe_b200")
        self.syn = importlib.import_module("midvision-probe_b200.synthetic")
        self.bb = importlib.import_module("midvision-probe_b200.backbones")
        self.models = {}
        self.dist = torch.distributed

    def init_device(self):
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
        # bind this rank's host threads (and the pinned staging buffers it allocates from here on) to the NUMA node of
        # its GPU: 8 ranks feeding their H2D copies from one node's cores and memory was what capped end-to-end scaling
        self.binding = self.mv.evaluation.bind_rank_to_gpu(self.local_rank, self.world)
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            self.dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def model(self, name):
        if name not in self.models:
            bb = self.bb
            self.models[name] = {"vit_multi": lambda: bb.DenseViT(bb.vit_b16(0), multilayer=True),
                                 "vit_last": lambda: bb.DenseViT(bb.vit_b16(0), multilayer=False),
                                 "resnet": lambda: bb.resnet50_layer4(0)}[name]().to(self.dev)
        return self.models[name]

    def pair(self, workload, i):
        """pair i of a workload (host tensors)."""
        if self.args.features == "gaussian":
            return {"navi": self.syn.navi_pair, "scannet": self.syn.scannet_pair, "spair": self.syn.spair_pair}[workload](i)
        if workload == "navi":
            return self.bb.navi_backbone_pair(i, self.model("vit_multi"), device=self.dev, noise=0.7)
        if workload == "scannet":
            return self.bb.scannet_backbone_pair(i, self.model("resnet"), device=self.dev, noise=1.0)
        return self.bb.spair_backbone_pair(i, self.model("vit_last"), device=self.dev, noise=0.5)


def cpu_pairs_per_s(ctx, workload, budget_s=12.0, max_pairs=6):
    """the CPU port of the reference (oracle/restated.py) on a bounded sample of the same workload."""
    from oracle import restated

    torch.set_num_threads(os.cpu_count() or 1)
    done, t_total = 0, 0.0
    for i in range(max_pairs):
        p = ctx.pair(workload, i)
        t0 = time.perf_counter()
        if workload == "navi":
            out = restated.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], NUM_CORR)
            restated.pair_errors(out[0], out[1], p["Rt"], p["intrinsics"])
        else:
            out = restated.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), NUM_CORR)
            restated.pair_errors(out[0], out[1], p["Rt"], p["K"])
        dt = time.perf_counter() - t0
        if i == 0 and max_pairs > 1:
            continue  # warm-up pair (thread pool, allocator)
        done += 1
        t_total += dt
        if t_total > budget_s:
            break
    return {"value": done / t_total, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{done} pairs of the same workload through oracle/restated.py (CPU fp32 torch port, exact brute-force k-NN)"}


DUMP_MAX_BYTES = 64 << 20


def write_outputs(ctx, dirname, prefix, arrays):
    """--dump-outputs: every array as dirname/<prefix>_<name>.npy (rank 0 only).  The inputs are seeded, so two builds
    run with the same arguments can be compared file by file."""
    import numpy as np

    if ctx.rank != 0:
        return
    ctx.dumped_bytes = getattr(ctx, "dumped_bytes", 0) + sum(a.nbytes for a in arrays.values())
    if ctx.dumped_bytes > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs would write {ctx.dumped_bytes} bytes (at most {DUMP_MAX_BYTES})")
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(dirname, f"{prefix}_{name}.npy"), a)


def dense_outputs(last, pool_dev, pool_ids, acc):
    """The matches a caller of the timed path holds after its last step: per pair the selected (query row, target row,
    weight, mutual-NN flag) of mv_k3_topk_matches, entries past the pair's live match count set to -1, and the recall hit
    counters of the whole timed region.  A lane of the CUDA-graph pipeline overwrites its results with its next pair, so
    of the last step the last pair of every lane is still held (all pairs without the graph): those are written."""
    import numpy as np

    held = {}
    for j, (p, r) in enumerate(last):
        held[id(r)] = (j, p, r)
    rows = sorted(held.values(), key=lambda x: x[0])
    k = max(max(r.k, 1) for _, _, r in rows)
    src, dst, wgt, mut = (np.full((len(rows), k), -1.0, dtype=dt) for dt in (np.float64, np.float64, np.float32, np.float32))
    count, pair, pos = (np.zeros(len(rows)) for _ in range(3))
    for i, (j, p, r) in enumerate(rows):
        n = int(r.k_dev.item())
        sel = r.sel_src[:n].long()
        src[i, :n] = sel.cpu().numpy()
        dst[i, :n] = r.sel_dst[:n].cpu().numpy()
        wgt[i, :n] = r.sel_weight[:n].cpu().numpy()
        mut[i, :n] = r.mutual[sel].cpu().numpy()
        count[i] = n
        pair[i] = pool_ids[next(s for s, q in enumerate(pool_dev) if q is p)]
        pos[i] = j
    return {"pair": pair, "position_in_step": pos, "match_count": count, "sel_src": src, "sel_dst": dst, "sel_weight": wgt,
            "sel_mutual": mut, "hits": acc.hits.cpu().double().numpy()}


# --------------------------------------------------------------------------------------------------------------
# the two dense workloads (NAVI / ScanNet shaped)
# --------------------------------------------------------------------------------------------------------------
def run_dense(ctx, workload, steps, warmup, fixed_pairs=0, light=False, dump=None):
    """one dense workload -> record.  fixed_pairs > 0: strong scaling over a fixed seeded set (configs[3]).
    light: only the device-resident arm and the end-to-end helper arm (the secondary workloads of a default run).
    dump: directory that receives the matches of the timed region's last step (dense_outputs)."""
    args, mv, dev, world, rank = ctx.args, ctx.mv, ctx.dev, ctx.world, ctx.rank
    C_, ev, L = mv.correspondence, mv.evaluation, mv._lib
    hbm_peak, tc_peak, tc_sustained, peak_kind = peaks()
    thr3, thr2 = THR[workload]
    big = ("feat_0", "feat_1", "xyz_grid_0", "xyz_grid_1", "depth_0", "depth_1")  # Rt / K are small host parameters, like in the callers
    fdt = torch.bfloat16 if args.feat_dtype == "bf16" else torch.float32

    def shaped(p):
        for k in ("feat_0", "feat_1"):
            if fdt != torch.float32:
                p[k] = p[k].to(fdt)
            if args.feat_layout == "hwc":
                p[k] = p[k].permute(1, 2, 0).contiguous().permute(2, 0, 1)  # same (C, h, w) tensor, channel-last memory
        return p

    # weak scaling: pool pair j of this rank is global pair rank + j * world (pair i lives on rank i mod world);
    # a fixed set is defined globally -- global pair i uses pool pair i mod POOL -- so that every N sees the same set
    pool_ids = list(range(POOL)) if fixed_pairs else [rank + j * world for j in range(POOL)]
    pool_host = [shaped(ctx.pair(workload, i)) for i in pool_ids]

    def pin(v):
        if v.dim() == 3 and not v.is_contiguous():  # keep the channel-last strides in pinned memory
            return v.permute(1, 2, 0).contiguous().pin_memory().permute(2, 0, 1)
        return v.pin_memory()

    pool_dev = [{k: (v.to(dev) if k in big else v) for k, v in p.items()} for p in pool_host]
    acc = ev.RecallAccumulator(thr3, thr2, device=dev)
    navi = workload == "navi"
    gk = ("xyz_grid_0", "xyz_grid_1", "intrinsics") if navi else ("depth_0", "depth_1", "K")

    def pair_eager(p):
        if navi:
            return ev.match_and_score_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], p["intrinsics"], p["Rt"], NUM_CORR, acc, sync=False)
        return ev.match_and_score_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"], p["Rt"], NUM_CORR, acc, sync=False)

    gm = None
    if not args.no_graph:
        p0 = pool_dev[0]
        gm = ev.PairPipeline("xyz" if navi else "depth", tuple(p0["feat_0"].shape), tuple(p0[gk[0]].shape),
                             NUM_CORR, K=p0.get("K"), device=dev, lanes=args.lanes, feat_layout=args.feat_layout, feat_dtype=fdt)

    def pair_device(p, a=acc):
        if gm is None:
            return pair_eager(p)
        return gm.submit(p["feat_0"], p["feat_1"], p[gk[0]], p[gk[1]], a, p["Rt"], p[gk[2]])

    # the schedule of the timed region: step s = pairs [s * PPS, (s + 1) * PPS) of this rank
    if fixed_pairs:
        mine = list(ev.shard_pairs(fixed_pairs, rank, world))   # global indices i with i mod world == rank
        steps = max(1, (len(mine) + PAIRS_PER_STEP - 1) // PAIRS_PER_STEP)
        sched = [[pool_dev[i % POOL] for i in mine[s * PAIRS_PER_STEP:(s + 1) * PAIRS_PER_STEP]] for s in range(steps)]
    else:
        sched = [[pool_dev[(s * PAIRS_PER_STEP + j) % POOL] for j in range(PAIRS_PER_STEP)] for s in range(steps)]

    def run_sched(which, a=acc, keep=False):
        """keep: -> [(pair, MatchResult)] of the last step (what --dump-outputs writes); without it no result is held,
        so that an eager (--no-graph) pass frees every pair's buffers as before"""
        which = list(which)
        for s in (which[:-1] if keep else which):
            for p in sched[s % len(sched)]:
                pair_device(p, a)
        return [(p, pair_device(p, a)) for p in sched[which[-1] % len(sched)]] if keep and which else []

    # ---------------- device-resident arm (value) ----------------
    run_sched(range(warmup))
    if gm is not None:
        gm.join()
    ctx.barrier()
    acc.hits.zero_()
    L.LAUNCHES["count"] = 0
    sampler = ClockSampler(ctx.local_rank).start()
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = run_sched(range(steps), keep=bool(dump))
    if gm is not None:
        gm.join()
    acc.all_reduce()  # the path's only collective: int64 hit counts
    e1.record()
    ctx.barrier()
    clocks = sampler.stop()
    if dump:
        write_outputs(ctx, dump, workload, dense_outputs(last, pool_dev, pool_ids, acc))
    launches = L.LAUNCHES["count"]
    ms_total = ctx.max_over_ranks(e0.elapsed_time(e1))
    summary = acc.summary()
    hits_vec = acc.hits.tolist()
    pairs_total = fixed_pairs if fixed_pairs else world * steps * PAIRS_PER_STEP
    value = pairs_total / (ms_total * 1e-3)

    # kernel 2's own duration: CUDA events around every mv_k2_sim_top2 call over the same steps, launched eagerly
    # (event records cannot be captured into the graph); same stream, same inputs, same L2 regime
    C_._PROFILE["k2_events"] = []
    k2_steps = max(1, min(steps, 10))
    lib = L.load()
    k2_cap = 2 * k2_steps * PAIRS_PER_STEP  # room for the Gram launch of the low-rank proposal next to the main product
    lib.mv_k2_profile_begin(k2_cap)  # event pairs right around the tcgen05 kernel inside the library
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for s in range(k2_steps):
        for p in sched[s % len(sched)]:
            pair_eager(p)
    e3.record()
    torch.cuda.synchronize()
    ms_eager = e2.elapsed_time(e3)
    k2_ev = C_._PROFILE.pop("k2_events")
    import ctypes

    kbuf = (ctypes.c_float * k2_cap)()
    dbuf = (ctypes.c_int * (3 * k2_cap))()
    n_k = lib.mv_k2_profile_read(kbuf, k2_cap)
    lib.mv_k2_profile_dims(dbuf, k2_cap)
    lib.mv_k2_profile_begin(0)
    # the main product's launches are the ones with the (n_max, C) of the calls match_rows made; with the low-rank proposal
    # the same kernel also computes the small Gram matrix of the source pixels (mv_k2_affinity): reported separately
    main_dims = {(n_, c_) for _, _, (n_, m_, c_, nd, md) in k2_ev}
    k2_kernel_ms = [kbuf[i] for i in range(max(n_k, 0)) if (dbuf[3 * i], dbuf[3 * i + 2]) in main_dims]
    gram = [(kbuf[i], dbuf[3 * i], dbuf[3 * i + 1], dbuf[3 * i + 2]) for i in range(max(n_k, 0)) if (dbuf[3 * i], dbuf[3 * i + 2]) not in main_dims]
    k2_call_ms = [a.elapsed_time(b) for a, b, _ in k2_ev]
    k2_kernel_ms = k2_kernel_ms[:len(k2_call_ms)]
    k2_ms = k2_kernel_ms if len(k2_kernel_ms) == len(k2_call_ms) and k2_kernel_ms else k2_call_ms
    k2_flops = [2.0 * (int(nd.item()) if nd is not None else n_) * (int(md.item()) if md is not None else m_) * c_
                for _, _, (n_, m_, c_, nd, md) in k2_ev]

    rec = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "strong" if fixed_pairs else "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME[workload], "pairs_per_step": PAIRS_PER_STEP, "pool_pairs": POOL,
                   "l2": "inputs larger than L2: 16 distinct pairs cycled, ~190 MB (NAVI) / ~330 MB (ScanNet) of features + rows touched per pair vs 126 MB L2",
                   "k2_cluster": args.cluster, "cuda_graph": gm is not None, "pairs_in_flight": args.lanes if gm is not None else 1,
                   "features": FEATURES_NAME[args.features], "feat_layout": args.feat_layout, "feat_dtype": args.feat_dtype,
                   "k2_operands": {"f16": "fp16, target rows centred (f16c)", "bf16": "bf16", "tf32": "tf32"}[args.dtype]},
        "clocks": clocks,
        "gpu_launches": launches,
        "recall": {"scored": summary["scored"], "recall_3d": summary["recall_3d"], "recall_2d": summary["recall_2d"], "mutual": summary["mutual"]},
    }
    if fixed_pairs:
        rec["config"]["fixed_set"] = {"pairs": fixed_pairs, "assignment": "pair i -> rank i mod N (evaluate_navi_correspondence.py:178-212 loop, sharded)"}
        rec["hits"] = hits_vec
        rec["hits_sha1"] = hashlib.sha1(json.dumps(hits_vec).encode()).hexdigest()
    if k2_ms:
        k2_avg_ms = sum(k2_ms) / len(k2_ms)
        k2_avg_flop = sum(k2_flops) / len(k2_flops)
        achieved = k2_avg_flop / (k2_avg_ms * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "k2_traffic.json")
        lowrank_used = bool(k2_ev) and k2_ev[0][2][2] < pool_dev[0]["feat_0"].shape[0]
        if os.path.exists(tpath) and args.dtype != "tf32":
            traffic = json.load(open(tpath)).get(workload + ("_lowrank" if lowrank_used else ""), {}).get("dram_bytes")
        # burst figure unless the timed pass is seconds long (the sustained cuBLAS figure is a 4 s back-to-back run)
        long_pass = ms_total > 2000.0
        peak = tc_sustained if long_pass else tc_peak
        rec["roofline"] = {
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": traffic,
            "traffic_note": "dram read+write bytes per launch from the committed ncu --set full capture of this shape (profiles/k2_traffic.json)",
            "peak_kind": f"{peak_kind} {'sustained' if long_pass else 'burst'} bf16 (timed pass {ms_total:.0f} ms)",
            "frac_burst": achieved / tc_peak, "frac_sustained": achieved / tc_sustained,
            "kernel": "k2_sim_top2_kernel alone (CUDA event pair recorded inside mv_k2_sim_top2_ld right around the launch, mv_k2_profile_*)",
            "launches_timed": len(k2_ms), "avg_ms": k2_avg_ms, "flop_per_launch": k2_avg_flop,
            "call_avg_ms": sum(k2_call_ms) / max(len(k2_call_ms), 1),
            "call_note": "call_avg_ms = event pair around the whole mv_k2_sim_top2_ld call: col_best memset + the kernel + the row-merge kernel (round 1's figure)",
            "k2_share_of_step": (sum(k2_ms) / k2_steps) / (ms_total / steps) if ms_total else None,
            "timed_in": "second, eagerly launched pass over the same steps (events cannot be recorded inside the captured graph)",
            "eager_pass_ms_per_step": ms_eager / k2_steps,
            "whole_step_tensor_frac": (k2_avg_flop * pairs_total / world / (ms_total * 1e-3) / 1e12) / tc_peak}
        Ck_main = k2_ev[0][2][2]
        C_feat = pool_dev[0]["feat_0"].shape[0]
        if Ck_main < C_feat:  # the low-rank proposal: kernel 2 multiplies over the target's source pixels, not the channels
            rec["roofline"]["lowrank"] = {
                "k2_columns": Ck_main, "channels": C_feat,
                "note": "kernel 2 ranks the same cosine similarities as a product over the target image's h*w source pixels (+8 "
                        "augmentation columns) instead of the C channels (csrc/lr_gram.cu); achieved / frac above count the FLOPs "
                        "ISSUED (2 n m k2_columns); at this K the kernel is bound by its epilogue (row top-2 + column arg-max of "
                        "every 128 x 256 tile), not by the tensor pipe",
                "dense_equivalent_tflops": achieved * (C_feat + 8) / Ck_main,
                "gram_launch": ({"avg_ms": sum(g[0] for g in gram) / len(gram), "rows": gram[0][1], "K": gram[0][3], "launches": len(gram)}
                                if gram else None)}
    if fixed_pairs and light:
        del gm
        return rec

    # ---------------- end-to-end arms: the reference-facing helper with host tensors ----------------
    pool_pin = [{k: (pin(v) if torch.is_tensor(v) else v) for k, v in p.items()} for p in pool_host]

    def call_helper(p):
        if navi:
            return C_.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], NUM_CORR)
        return C_.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), NUM_CORR)

    def time_helper(pool, n_calls, n_warm=8):
        for j in range(n_warm):
            out = call_helper(pool[j % POOL])
        ctx.barrier()
        t0 = time.perf_counter()
        for j in range(n_calls):
            out = call_helper(pool[j % POOL])
        torch.cuda.synchronize()
        return world * n_calls / ctx.max_over_ranks(time.perf_counter() - t0), out

    e2e_steps = max(2, min(steps, 20) // 2)
    n_calls = e2e_steps * PAIRS_PER_STEP
    e2e_value, out = time_helper(pool_pin, n_calls)
    h2d = PAIRS_PER_STEP * sum(pool_host[0][k].numel() * pool_host[0][k].element_size() for k in big if k in pool_host[0])
    d2h = PAIRS_PER_STEP * sum(o.numel() * o.element_size() for o in out)
    rec["e2e"] = {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                  "host_memory": "pinned",
                  "api": "correspondence.estimate_correspondence_xyz(host tensors)" if navi else "correspondence.estimate_correspondence_depth(host tensors)"}
    # the same helper fed PAGEABLE host tensors -- what the reference's callers hold (.detach().cpu(), navi:149-150)
    pool_page = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in p.items()} for p in pool_host]
    pg_value, _ = time_helper(pool_page, max(PAIRS_PER_STEP, n_calls // 2))
    rec["e2e_pageable"] = {"value": pg_value, "unit": "pairs/s", "host_memory": "pageable (plain torch tensors, as the reference's callers hold them)",
                           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
    if light:
        del gm
        return rec

    # the same helper fed 16-bit feature maps from pinned memory -- what a backbone under bf16 autocast hands over (the helper
    # uploads them as they are and widens them exactly on the device: tests/test_gpu_pipeline.py::test_16bit_feature_maps_*):
    # half the PCIe bytes of the fp32 arm.  Informational: the headline e2e above is the fp32 hand-over of the reference.
    if args.feat_dtype == "f32":
        pool_16 = [{k: (pin(v.to(torch.bfloat16)) if (torch.is_tensor(v) and k in ("feat_0", "feat_1")) else (pin(v) if torch.is_tensor(v) else v))
                    for k, v in p.items()} for p in pool_host]
        v16, _ = time_helper(pool_16, max(PAIRS_PER_STEP, n_calls // 2))
        rec["e2e_bf16_features"] = {"value": v16, "unit": "pairs/s", "host_memory": "pinned, bf16 feature maps (autocast backbone)",
                                    "h2d_bytes_per_step": h2d - PAIRS_PER_STEP * sum(pool_host[0][k].numel() * 2 for k in ("feat_0", "feat_1"))}

    # the same synchronous helper with DEVICE-resident tensors (a caller that keeps the backbone output on the GPU,
    # SURVEY 8f.1): no upload, results stay on the device, one host sync per call for the match count
    hd_value, _ = time_helper(pool_dev, n_calls, n_warm=4)
    rec["helper_device_tensors"] = {"value": hd_value, "unit": "pairs/s",
                                    "api": "the same helper called with device-resident tensors (no H2D; results returned on the device)"}
    # the same host-resident pairs through the pair pipeline (the evaluation loop's API: submit / join, integer hit
    # counts read back once at the end): the upload of one pair overlaps the kernels of the previous ones
    if gm is not None:
        acc2 = ev.RecallAccumulator(thr3, thr2, device=dev)

        def step_pipe(s):
            for j in range(PAIRS_PER_STEP):
                p = pool_pin[(s * PAIRS_PER_STEP + j) % POOL]
                gm.submit(p["feat_0"], p["feat_1"], p[gk[0]], p[gk[1]], acc2, p["Rt"], p[gk[2]])

        for s in range(2):
            step_pipe(s)
        gm.join()
        ctx.barrier()
        acc2.hits.zero_()
        t0 = time.perf_counter()
        for s in range(e2e_steps):
            step_pipe(s)
        gm.join()
        counts = acc2.hits.cpu()  # device -> host read of the result, inside the timed region
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        rec["e2e_pipeline"] = {"value": world * e2e_steps * PAIRS_PER_STEP / dt, "unit": "pairs/s",
                               "api": "evaluation.PairPipeline.submit(host tensors) + RecallAccumulator read-back",
                               "scored": int(counts[0]), "d2h_bytes_total": counts.numel() * 8}
    # the frozen backbone next to the matching path: forward of both images on this GPU (PyTorch, fp32 like the
    # reference), features handed to the pair pipeline on the device (no CPU round trip, SURVEY 8f.1)
    if args.features == "backbone":
        rec["backbone"] = backbone_record(ctx, workload, gm, pool_dev, gk, acc)
    del gm
    return rec


def backbone_record(ctx, workload, gm, pool_dev, gk, acc):
    bb, dev = ctx.bb, ctx.dev
    model = ctx.model("vit_multi" if workload == "navi" else "resnet")
    H, W = (448, 448) if workload == "navi" else (480, 640)
    imgs = [bb._pair_images(100 + i, H, W, True, 0.5).to(dev) for i in range(4)]

    def fwd(x, autocast):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            return model.features(x)

    out = {}
    for name, autocast in (("fp32", False), ("bf16_autocast", True)):
        for x in imgs[:2]:
            fwd(x, autocast)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 8
        for i in range(n):
            fwd(imgs[i % 4], autocast)
        e1.record()
        torch.cuda.synchronize()
        out[f"forward_ms_per_pair_{name}"] = e0.elapsed_time(e1) / n
    if gm is not None:
        # backbone forward + matching, features stay on the device: the pair pipeline is fed the backbone's output
        p0 = pool_dev[0]
        n = 48
        for i in range(4):
            f = fwd(imgs[i % 4], False).float()
            gm.submit(f[0], f[1], p0[gk[0]], p0[gk[1]], acc, p0["Rt"], p0[gk[2]])
        gm.join()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n):
            f = fwd(imgs[i % 4], False).float()
            p = pool_dev[i % POOL]
            gm.submit(f[0], f[1], p[gk[0]], p[gk[1]], acc, p["Rt"], p[gk[2]])
        gm.join()
        torch.cuda.synchronize()
        out["pairs_per_s_with_backbone"] = ctx.world * n / ctx.max_over_ranks(time.perf_counter() - t0)
    out["model"] = "random-init ViT-B/16 @448, blocks [2,5,8,11] concat" if workload == "navi" else "random-init ResNet-50 layer4 @480x640"
    out["note"] = "PyTorch forward of both images of a pair on the same GPU (fp32 matmuls, torch's default TF32 convolutions); matching fed on the device"
    return out


# --------------------------------------------------------------------------------------------------------------
# kernel 1 alone
# --------------------------------------------------------------------------------------------------------------
def k1_record(ctx):
    """kernel 1 on one image of each dense workload, timed with CUDA events: a CUDA graph of 24 launches writing to 6
    rotating output sets (> L2).  Bytes: `surveyed` = C*h*w*4 + n*C*2 (SURVEY 8d: the map read + ONE 16-bit row plane),
    `moved` = what this build really moves (two 16-bit planes: the fp16 operand rows and their residual for kernel 3)."""
    from ctypes import c_void_p

    mv, dev = ctx.mv, ctx.dev
    C_, L = mv.correspondence, mv._lib
    hbm_peak, _, _, peak_kind = peaks()
    out = {}
    for kind in ("navi", "scannet"):
        p = ctx.pair(kind, 0)
        f = p["feat_0"].to(dev)
        calls = []
        orig_call = L.call

        def spy(name, *a):
            if name in ("mv_k1_sample_f16c", "mv_k1_sample_normalize", "mv_k1_grid_f16c"):
                calls.append((name, a))
            return orig_call(name, *a)

        L.call = spy
        try:
            fm0, fm1, kw0, kw1 = C_._pair_maps(f, p["feat_1"].to(dev), dev)
            if kind == "navi":
                s = C_.prepare_xyz_side(fm0, p["xyz_grid_0"].to(dev), dev, sync=True, **kw0)
            else:
                Kh, Kinv = C_._host_mat(p["K"]), C_._host_mat(p["K"].inverse())
                s = C_.prepare_depth_side(fm0, p["depth_0"].to(dev), Kh, Kinv, dev, sync=True, **kw0)
        finally:
            L.call = orig_call
        name, a = calls[0]
        n, C, h, w = s.n, fm0[1], fm0[2], fm0[3]
        f16 = name != "mv_k1_sample_normalize"
        t16 = torch.float16 if f16 else torch.bfloat16
        pitch = L.f16c_pitch(C) if f16 else C
        sets = [(torch.empty((n, pitch), dtype=t16, device=dev), torch.empty((n, C), dtype=t16, device=dev)) for _ in range(6)]
        # positions of the (stream, 16-bit rows, residual rows) arguments of the recorded call
        slots = {"mv_k1_sample_f16c": (-1, 13, 15), "mv_k1_sample_normalize": (-1, 9, 10), "mv_k1_grid_f16c": (-1, 10, 12)}[name]
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            def launch(i):
                hi, lo = sets[i % 6]
                b = list(a)
                b[slots[0]], b[slots[1]], b[slots[2]] = c_void_p(st.cuda_stream), L.ptr(hi), L.ptr(lo)
                L.call(name, *b)
            launch(0)
            st.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                for i in range(24):
                    launch(i)
            g.replay()
            st.synchronize()
            ts = []
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                g.replay()
                e1.record(st)
                st.synchronize()
                ts.append(e0.elapsed_time(e1) / 24 * 1e3)
        us = statistics.median(ts)
        surveyed = C * h * w * 4 + n * C * 2
        moved = C * h * w * 4 + n * ((C + 8 if f16 else C) + C) * 2
        out[f"{kind}_side"] = {
            "points": n, "C": C, "entry_point": name, "mode": "bicubic 4x (28x28 -> live pixels of 112x112)" if kind == "navi" else "bilinear (15x20 -> 120x160 depth pixels)",
            "avg_us": us, "bytes_surveyed": surveyed, "bytes_moved": moved,
            "GB/s_surveyed": surveyed / us / 1e3, "GB/s_moved": moved / us / 1e3, "peak": hbm_peak, "peak_kind": f"{peak_kind} copy bandwidth (read + write)",
            "frac_surveyed": surveyed / us / 1e3 / hbm_peak, "frac_moved": moved / us / 1e3 / hbm_peak,
            "note": "the kernel only writes to HBM (the 2.5-9.6 MB map stays in L2); a write-only stream (cudaMemset) reaches ~3.9 TB/s on this part, "
                    "which is the practical roof of frac_moved (~0.6)",
            "timed": "CUDA events on the launching stream around a CUDA graph of 24 launches, 6 rotating output sets (> L2), median of 5"}
        del sets, s
    return out


# --------------------------------------------------------------------------------------------------------------
# SPair (configs[0])
# --------------------------------------------------------------------------------------------------------------
SPAIR_DRAM_BYTES_PER_PAIR = 1.441e6  # ncu --set full of one 2368-pair launch (dram__bytes_read.sum + dram__bytes_write.sum) / pairs
SPAIR_BATCH = 2368  # pairs per step (one launch) = 8 per CTA at 2 CTAs x 148 SMs; 1.2 MB of features per pair -> 2.85 GB per step
SPAIR_BATCH_E2E = 1184  # pairs per step of the end-to-end arm (1.4 GB of pinned host memory per rank)


def run_spair(ctx, steps, warmup, dump=None):
    """SPair-shaped pairs, (2, 768, 14, 14) features + 20 key points, a step = SPAIR_BATCH pairs through
    spair.compute_errors_batch (one fused launch).  HBM-bound: the roofline figure is the feature bytes read per launch.
    dump: directory that receives the four (B, K) results of the last timed launch and the PCK counts."""
    mv, dev, world, rank = ctx.mv, ctx.dev, ctx.world, ctx.rank
    sp, L = mv.spair, mv._lib
    hbm_peak, _, _, peak_kind = peaks()
    base = [ctx.pair("spair", rank + world * i) for i in range(32)]
    B, Bh = SPAIR_BATCH, SPAIR_BATCH_E2E
    pick = lambda key: torch.stack([torch.as_tensor(base[i % 32][key]) for i in range(Bh)])
    host = {"feats": pick("feats").pin_memory(), "kps_i": pick("kps_i").pin_memory(), "kps_j": pick("kps_j").pin_memory(),
            "ts": pick("thresh_scale").float().pin_memory()}
    # the device-resident batch: the same 32 distinct pairs cycled B times, gathered on the device
    idx = torch.arange(B, device=dev) % 32
    d = {k: v[:32].to(dev)[idx].contiguous() for k, v in host.items()}
    hits = torch.zeros(2, dtype=torch.int64, device=dev)

    def step(src):
        return sp.compute_errors_batch(src["feats"], src["kps_i"], src["kps_j"], src["ts"], 224, hits=hits)

    for _ in range(warmup):
        step(d)
    ctx.barrier()
    hits.zero_()
    L.LAUNCHES["count"] = 0
    sampler = ClockSampler(ctx.local_rank).start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps - 1):
        step(d)
    last = step(d)
    if world > 1:
        ctx.dist.all_reduce(hits, op=ctx.dist.ReduceOp.SUM)  # the path's only collective: PCK counts
    e1.record()
    ctx.barrier()
    clocks = sampler.stop()
    if dump:
        names = ("error_same", "error_nn", "index_nn", "pred")
        arrays = {nm: t.cpu().to(torch.float32 if t.is_floating_point() else torch.float64).numpy() for nm, t in zip(names, last)}
        write_outputs(ctx, dump, "spair", dict(arrays, hits=hits.cpu().double().numpy()))
    launches = L.LAUNCHES["count"]
    ms_total = ctx.max_over_ranks(e0.elapsed_time(e1))
    value = world * steps * B / (ms_total * 1e-3)
    h = hits.tolist()
    # end to end: pinned host tensors in, the four (B, K) result tensors back on the host, every step
    for _ in range(2):
        out = step(host)
    ctx.barrier()
    t0 = time.perf_counter()
    e2e_steps = max(2, steps // 2)
    for _ in range(e2e_steps):
        out = [o.cpu() for o in step(host)]
    torch.cuda.synchronize()
    e2e = world * e2e_steps * Bh / ctx.max_over_ranks(time.perf_counter() - t0)
    byts = d["feats"].numel() * 4
    per_launch_ms = ms_total / steps
    # the same launches with one tf32 MMA per heat-map tile instead of three (spair.set_heatmap_precision("tf32"): arg-max parity
    # at a 1e-3 heat-map gap instead of 1e-5) -- informational, the headline stays the 3xTF32 default
    sp.set_heatmap_precision("tf32")
    try:
        for _ in range(2):
            step(d)
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for _ in range(steps):
            step(d)
        t1e.record()
        torch.cuda.synchronize()
        ms_1x = ctx.max_over_ranks(t0e.elapsed_time(t1e)) / steps
    finally:
        sp.set_heatmap_precision("3xtf32")
    rec = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": per_launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME["spair"], "pairs_per_step": B, "pairs_per_e2e_step": Bh,
                   "l2": "inputs larger than L2: 2.85 GB of features per step",
                   "features": FEATURES_NAME[ctx.args.features].replace("blocks [2,5,8,11] concat / ResNet-50 layer4", "last block @224")},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in host.values()),
                "d2h_bytes_per_step": sum(o.numel() * o.element_size() for o in out), "steps": e2e_steps,
                "api": "spair.compute_errors_batch(host tensors)"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": byts / (per_launch_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": byts / (per_launch_ms * 1e-3) / 1e9 / hbm_peak, "traffic": SPAIR_DRAM_BYTES_PER_PAIR * B,
                     "peak_kind": f"{peak_kind} copy bandwidth",
                     "kernel": "spair_stream_kernel (one launch per step; algorithmic bytes = the (B, 2, C, h, w) features, read once; "
                               "traffic = dram__bytes_read + write of one launch under ncu, profiles/r2_spair_stream_final_2368.txt: image i is "
                               "read twice and its second read hits L2 only in part)",
                     "avg_ms": per_launch_ms, "bytes_per_launch": byts},
        "recall": {"keypoints_in_both": h[0], "pck_0.10": 100.0 * h[1] / max(h[0], 1)},
        "tf32_single_term": {"value": world * B / (ms_1x * 1e-3), "unit": "pairs/s", "frac_of_hbm_peak": byts / (ms_1x * 1e-3) / 1e9 / hbm_peak,
                             "note": "spair.set_heatmap_precision('tf32'): one tf32 MMA per tile, parity at a 1e-3 heat-map gap"},
    }
    if world == 1 and rank == 0 and not ctx.args.no_cpu_baseline:
        from oracle import restated

        torch.set_num_threads(os.cpu_count() or 1)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < 8.0:
            p = base[n % 32]
            restated.spair_compute_errors(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"])
            n += 1
        rec["cpu_baseline"] = {"value": n / (time.perf_counter() - t0), "unit": "pairs/s", "cores": torch.get_num_threads(),
                               "kind": "port", "sample": f"{n} pairs through oracle/restated.py spair_compute_errors (fp32 torch on the CPU)"}
    return rec


# --------------------------------------------------------------------------------------------------------------
# --impl reference
# --------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port), all host threads, on the same
    workload.  Honours --steps / --warmup; each step is a bounded sample (2 dense pairs / 64 SPair pairs) and a wall-time
    cap of REF_WALL_CAP_S keeps the run within minutes (`capped` says whether it cut the requested steps).  Under torchrun
    rank 0 alone runs it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    syn = importlib.import_module("midvision-probe_b200.synthetic")
    workload = "navi" if args.workload == "all" else args.workload
    per_step = 64 if workload == "spair" else 2
    torch.set_num_threads(os.cpu_count() or 1)
    from oracle import restated

    def one(p):
        if workload == "spair":
            restated.spair_compute_errors(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"])
        elif workload == "navi":
            out = restated.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], NUM_CORR)
            restated.pair_errors(out[0], out[1], p["Rt"], p["intrinsics"])
        else:
            out = restated.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), NUM_CORR)
            restated.pair_errors(out[0], out[1], p["Rt"], p["K"])

    # features: this arm never touches the GPU, so it takes the Gaussian maps of the same shapes; the reference path's
    # cost (dense fp32 GEMM + top-k + gathers + interpolation) does not depend on the feature values
    gen = {"navi": syn.navi_pair, "scannet": syn.scannet_pair, "spair": syn.spair_pair}[workload]
    pairs = [gen(i) for i in range(POOL)]  # inputs exist before the clock starts
    for w in range(args.warmup):
        one(pairs[w % len(pairs)])
    t1 = time.perf_counter()
    done = 0
    for s in range(args.steps):
        for j in range(per_step):
            one(pairs[(s * per_step + j) % len(pairs)])
        done += 1
        if time.perf_counter() - t1 > REF_WALL_CAP_S:
            break
    dt = time.perf_counter() - t1
    val = done * per_step / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / done, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME[workload], "pairs_per_step": per_step, "steps_requested": args.steps,
                   "capped": done < args.steps, "wall_cap_s": REF_WALL_CAP_S,
                   "note": "a step of this arm is a bounded sample of the step of the B200 arm (2 of its 32 pairs); pairs/s is per pair and comparable"},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{done * per_step} pairs, oracle/restated.py (fp32 torch CPU port of evals/utils/correspondence.py with exact brute-force k-NN in place of faiss-gpu)"},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def stress(ctx, tc_peak):
    """BASELINE.json configs[4]: 19200 x 19200 x 768 kernel 2 alone, timed in isolation (burst peak)."""
    from ctypes import c_size_t

    L, C_ = ctx.mv._lib, ctx.mv.correspondence
    n = m = 19200
    C = 768
    A, B = ctx.syn.stress_rows(0, n=n, m=m, C=C)
    out = {}
    for name, dt_flag in (("bf16", 0), ("f16", 2), ("tf32", 1)):
        t16 = {0: torch.bfloat16, 2: torch.float16}.get(dt_flag)
        Ad = (A.cuda().to(t16) if t16 else A.cuda()).contiguous()
        Bd = (B.cuda().to(t16) if t16 else B.cuda()).contiguous()
        rv = torch.empty(n, 2, device="cuda")
        ri = torch.empty(n, 2, dtype=torch.int32, device="cuda")
        cb = torch.empty(m, dtype=torch.int64, device="cuda")
        wsb = L.load().mv_k2_workspace_bytes(n, m)
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

        def launch():
            L.call("mv_k2_sim_top2", L.ptr(Ad), L.ptr(Bd), n, m, C, None, None, dt_flag, C_._CFG["cluster"], L.ptr(rv), L.ptr(ri),
                   L.ptr(cb), L.ptr(ws), c_size_t(wsb), C_._stream())

        for _ in range(3):
            launch()
        times = []
        for _ in range(10):
            flush.zero_()  # L2 flush between timed launches
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            launch()
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        ms = statistics.median(times)
        tf = 2.0 * n * m * C / (ms * 1e-3) / 1e12
        peak = tc_peak if dt_flag != 1 else tc_peak / 2
        out[name] = {"ms": ms, "tflops": tf, "frac_of_peak": tf / peak, "peak": peak, "l2": "flushed between launches"}
    return out


def h2d_link_probe(ctx, bytes_per_pair):
    """The ceiling of the end-to-end arm on THIS box at THIS N: all ranks copy one pair's worth of pinned host memory to their
    GPU at the same time, back to back; pairs/s ceiling = aggregate bandwidth / bytes per pair.  (On the 8-GPU boxes of this
    pool pairs of GPUs share a PCIe uplink: 54.9 GB/s alone, 29.8 GB/s each at N = 8 -- profiles/r2_h2d_scale.txt.)"""
    n = int(bytes_per_pair) // 4
    src = [torch.zeros(n, dtype=torch.float32).pin_memory() for _ in range(4)]
    dst = torch.empty(n, dtype=torch.float32, device=ctx.dev)
    for s_ in src:
        dst.copy_(s_, non_blocking=True)
    torch.cuda.synchronize()
    reps, best = 32, float("inf")
    for _ in range(5):  # best of five rounds: the figure is a ceiling, a descheduled host thread must not lower it
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(reps):
            dst.copy_(src[i % 4], non_blocking=True)
        torch.cuda.synchronize()
        best = min(best, ctx.max_over_ranks(time.perf_counter() - t0))
    agg = ctx.world * reps * n * 4 / best / 1e9
    return {"aggregate_GBps": agg, "per_gpu_GBps": agg / ctx.world, "pairs_per_s_ceiling": agg * 1e9 / (n * 4),
            "note": "all ranks copying from pinned host memory at once: what the PCIe topology of this box gives N GPUs"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of the headline workload (default 20); the ScanNet / SPair records of --workload all time "
                         "max(3, K // 4) / max(5, K // 2) steps, and --pairs sets its own count (the two do not combine)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "navi", "scannet", "spair"],
                    help="all (default) = NAVI headline + ScanNet / SPair / kernel-1 / sharded-set sub-records in the same line")
    ap.add_argument("--pairs", type=int, default=0,
                    help="strong scaling (BASELINE.json configs[3]): a FIXED seeded set of this many pairs of the headline workload, pair i on rank i mod N")
    ap.add_argument("--features", default="backbone", choices=["backbone", "gaussian"])
    ap.add_argument("--dtype", default="f16", choices=["f16", "bf16", "tf32"],
                    help="kernel 2 operand type: f16 = centred fp16 rows (default), bf16, tf32")
    ap.add_argument("--cluster", type=int, default=int(os.environ.get("MVMATCH_CLUSTER", "-1")),
                    help="kernel 2 cluster mode: -1 auto, 1 single CTA, 2 / 4 B-tile multicast, 20 CTA pair (cta_group::2)")
    ap.add_argument("--feat-dtype", default="f32", choices=["f32", "bf16"],
                    help="dtype of the feature tensors handed to the path: f32 = the reference's convention (BASELINE config); "
                         "bf16 = an autocast backbone's output, uploaded as 16-bit and widened on the device (supplementary)")
    ap.add_argument("--k1-only", action="store_true", help="print only the kernel-1 record (CUDA-event timing of kernel 1 alone) and exit")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stress", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying the captured CUDA graph")
    ap.add_argument("--lanes", type=int, default=6, help="pairs in flight on separate streams (CUDA-graph arm)")
    ap.add_argument("--feat-layout", default="chw", choices=["chw", "hwc"],
                    help="memory layout of the (C, h, w) feature tensors handed to the path: chw = contiguous, as the "
                         "reference's tokens_to_output returns them; hwc = channel-last views (ViT token order), no transpose kernel")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of each workload, write what its last step computed as DIR/<workload>_<name>.npy")
    args = ap.parse_args()
    if args.pairs and args.steps is not None:
        ap.error("--pairs P times ceil(P / N / 32) steps of its fixed set; it does not take --steps")
    args.steps = 20 if args.steps is None else args.steps
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return
    args.warmup = max(args.warmup, 3)
    ctx = Ctx(args)
    ctx.init_device()
    ctx.mv.correspondence.set_match_precision(dtype=args.dtype, cluster=args.cluster)
    _, tc_peak, _, _ = peaks()
    if args.k1_only:
        print(json.dumps({"k1": k1_record(ctx), "k1_grid": ctx.mv.correspondence._CFG["k1_grid"]}), flush=True)
        return
    head = "navi" if args.workload == "all" else args.workload
    dump = args.dump_outputs
    if head == "spair":
        line = run_spair(ctx, args.steps, args.warmup, dump=dump)
    else:
        line = run_dense(ctx, head, args.steps, args.warmup, fixed_pairs=args.pairs, dump=dump)
        if ctx.world == 1 and ctx.rank == 0 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_pairs_per_s(ctx, head)
    line["host_binding"] = ctx.binding
    if head != "spair" and "e2e" in line:
        line["e2e"]["h2d_link"] = h2d_link_probe(ctx, line["e2e"]["h2d_bytes_per_step"] / line["config"]["pairs_per_step"])
    if args.workload == "all":
        sub_steps = max(3, args.steps // 4)
        line["workloads"] = {"scannet": run_dense(ctx, "scannet", sub_steps, 3, light=True, dump=dump),
                             "spair": run_spair(ctx, max(5, args.steps // 2), 3, dump=dump)}
        if ctx.world == 1 and ctx.rank == 0 and not args.no_cpu_baseline:
            line["workloads"]["scannet"]["cpu_baseline"] = cpu_pairs_per_s(ctx, "scannet", budget_s=10.0, max_pairs=3)
        if not args.pairs:
            fs = run_dense(ctx, "navi", 0, 1, fixed_pairs=SHARDED_PAIRS, light=True)
            line["sharded_set"] = {"pairs": SHARDED_PAIRS, "assignment": "pair i -> rank i mod N", "hits": fs["hits"], "hits_sha1": fs["hits_sha1"],
                                   "pairs_per_s": fs["value"], "recall": fs["recall"],
                                   "note": "BASELINE.json configs[3] in small: the digest must be identical for every N (full size: --pairs 10000)"}
        if ctx.rank == 0:
            line["k1"] = k1_record(ctx)
    if ctx.world == 1 and ctx.rank == 0 and not args.no_stress:
        line["k2_stress"] = stress(ctx, tc_peak)
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)
    if ctx.world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
