"""Pair-sharded evaluation of the dense-correspondence benchmarks on one or more B200s.

Every image pair is independent (loops at evaluate_navi_correspondence.py:178,
render_scannet_correspondence.py:188, evaluate_spair_correspondence.py:108), so pair i runs on rank
i mod world; each rank accumulates integer hit counts on its device (mv_k3_score) and ONE NCCL
all-reduce of that small int64 vector at the end makes the recalls identical on every rank and equal
to the single-GPU run.  No other collective exists on this path.
"""
from ctypes import c_void_p

import torch

from . import _lib as L
from . import correspondence as C_

__all__ = ["RecallAccumulator", "shard_pairs", "match_and_score_depth", "match_and_score_xyz", "GraphedPairMatcher",
           "PairPipeline", "bind_rank_to_gpu"]


def _cpulist(text):
    out = []
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        out.extend(range(int(a), int(b or a) + 1))
    return out


def bind_rank_to_gpu(local_rank, local_world=1):
    """Pin this process (one per GPU) to a share of the cores of its GPU's NUMA node, BEFORE it allocates pinned
    staging memory, so that the host side of its H2D copies (page-locked buffers, the memcpy into them, the launch
    thread) lives next to the PCIe root of its own GPU instead of on node 0 with every other rank.

    The node comes from /sys/bus/pci/devices/<bus id>/numa_node, its cores from /sys/devices/system/node/nodeK/cpulist;
    ranks that share a node split its cores evenly.  Memory follows by first touch (and set_mempolicy when libnuma's
    syscall is reachable).  Returns a description dict; never raises (a box without the sysfs files is left unbound)."""
    import ctypes
    import os

    info = {"bound": False}
    try:
        import torch.cuda as tc

        ngpu = tc.device_count()
        nodes = []
        for g in range(ngpu):
            bus = tc.get_device_properties(g).pci_bus_id if hasattr(tc.get_device_properties(g), "pci_bus_id") else None
            dom = getattr(tc.get_device_properties(g), "pci_domain_id", 0)
            dev_id = getattr(tc.get_device_properties(g), "pci_device_id", 0)
            path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/numa_node" if bus is not None else None
            node = -1
            if path and os.path.exists(path):
                node = int(open(path).read().strip())
            nodes.append(node)
        node = nodes[local_rank] if local_rank < len(nodes) else -1
        if node < 0:
            all_nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
            if len(all_nodes) <= 1:
                info["reason"] = "single NUMA node"
                return info
            node = all_nodes[local_rank * len(all_nodes) // max(local_world, 1) % len(all_nodes)]
        cpus = _cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read())
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0))) or cpus
        peers = [r for r in range(min(local_world, max(len(nodes), 1))) if (nodes[r] if r < len(nodes) else -1) == nodes[local_rank]] if nodes else [local_rank]
        if local_rank not in peers:
            peers = [local_rank]
        share = max(1, len(allowed) // len(peers))
        k = peers.index(local_rank)
        mine = allowed[k * share:(k + 1) * share] or allowed
        os.sched_setaffinity(0, mine)
        info.update({"bound": True, "numa_node": node, "cpus": f"{mine[0]}-{mine[-1]}", "n_cpus": len(mine), "ranks_on_node": len(peers)})
        try:  # prefer this node for every later allocation (MPOL_PREFERRED = 1); best effort
            libc = ctypes.CDLL(None, use_errno=True)
            mask = ctypes.c_ulong(1 << node)
            rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(64))  # __NR_set_mempolicy on x86-64
            info["mempolicy"] = "preferred" if rc == 0 else f"errno {ctypes.get_errno()}"
        except Exception as e:  # noqa: BLE001
            info["mempolicy"] = f"unavailable ({type(e).__name__})"
    except Exception as e:  # noqa: BLE001 -- binding is an optimisation, never a failure
        info["reason"] = f"{type(e).__name__}: {e}"
    return info


def shard_pairs(num_pairs, rank, world):
    """indices of the pairs this rank owns (round-robin keeps variable-size pairs balanced)."""
    return range(rank, num_pairs, world)


class RecallAccumulator:
    """Integer hit counters for 3-D (metres) and 2-D (pixels) thresholds.

    Layout of ``hits`` (include/mvmatch.h, mv_k3_score): [scored, mutual, 3d[n3], 2d[n2],
    mutual&3d[n3], mutual&2d[n2]].  recall = 100 * hits / scored reproduces
    ``100 * (err < th).float().mean()`` (evaluate_navi_correspondence.py:200-212,
    render_scannet_correspondence.py:253-264) without floating-point accumulation.
    """

    def __init__(self, thr3d, thr2d, device=None, angle_bins=None, bin_threshold=0.02):
        """angle_bins: optional edges in degrees (e.g. [0, 30, 60, 90, 120]); every scored pair then also adds its
        (#err3d < bin_threshold, #matches) to the bin of its relative rotation angle -- the integer form of
        compute_binned_performance(rec_2cm, rel_ang, bins) (evaluate_navi_correspondence.py:214-223; identical to
        the reference's mean of per-pair recalls whenever every pair yields the same number of matches, which
        the reference's torch.stack requires)."""
        if len(thr3d) > L.MV_MAX_THRESHOLDS or len(thr2d) > L.MV_MAX_THRESHOLDS:
            raise ValueError(f"at most {L.MV_MAX_THRESHOLDS} thresholds per list")
        self.thr3d = [float(t) for t in thr3d]
        self.thr2d = [float(t) for t in thr2d]
        self.n3, self.n2 = len(self.thr3d), len(self.thr2d)
        self.device = device
        self.hits = torch.zeros(2 + 2 * (self.n3 + self.n2), dtype=torch.int64, device=device)
        self._t3 = L.host_floats(self.thr3d) if self.n3 else None
        self._t2 = L.host_floats(self.thr2d) if self.n2 else None
        self.angle_bins = [float(a) for a in angle_bins] if angle_bins is not None else None
        self.bin_threshold = float(bin_threshold)
        self._tb = L.host_floats([self.bin_threshold])
        nb = len(self.angle_bins) - 1 if self.angle_bins else 0
        # per bin the 4 counters mv_k3_score writes for one 3-D threshold: [scored, mutual, hits, mutual&hits]
        self.bin_hits = torch.zeros((max(nb, 1), 4), dtype=torch.int64, device=device)

    def score(self, match, xyz0, xyz1, Rt, K, want_errors=False):
        """Accumulate the counts of one pair. Rt: (3|4, 4), K: (3, 3) host or device tensors."""
        dev = xyz0.device
        Rt_h = L.host_floats(Rt.detach().float().cpu()[:3, :4].reshape(-1).tolist())
        K_h = L.host_floats(K.detach().float().cpu().reshape(-1).tolist())
        k = match.k
        e3 = torch.empty((max(k, 1),), dtype=torch.float32, device=dev) if want_errors else None
        e2 = torch.empty((max(k, 1),), dtype=torch.float32, device=dev) if want_errors else None
        L.call("mv_k3_score", L.ptr(match.sel_src), L.ptr(match.sel_dst), L.ptr(match.k_dev), k, L.ptr(xyz0),
               L.ptr(xyz1), L.ptr(match.mutual), Rt_h, K_h, self._t3, self.n3, self._t2, self.n2, None, None,
               L.ptr(e3), L.ptr(e2), L.ptr(self.hits), C_._stream())
        if self.angle_bins:
            from .transformations import so3_rotation_angle

            ang = float(so3_rotation_angle(Rt.detach().float().cpu()[None, :3, :3])[0]) * 180.0 / 3.141592653589793
            for b in range(len(self.angle_bins) - 1):
                if self.angle_bins[b] <= ang < self.angle_bins[b + 1]:
                    L.call("mv_k3_score", L.ptr(match.sel_src), L.ptr(match.sel_dst), L.ptr(match.k_dev), k, L.ptr(xyz0),
                           L.ptr(xyz1), L.ptr(match.mutual), Rt_h, K_h, self._tb, 1, None, 0, None, None, None, None,
                           c_void_p(self.bin_hits.data_ptr() + 32 * b), C_._stream())
                    break
        return (e3, e2) if want_errors else None

    def all_reduce(self):
        """Sum the counters over all ranks (the path's only collective)."""
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            torch.distributed.all_reduce(self.hits, op=torch.distributed.ReduceOp.SUM)
            if self.angle_bins:
                torch.distributed.all_reduce(self.bin_hits, op=torch.distributed.ReduceOp.SUM)
        return self

    def binned_recall(self):
        """[100 * hits / scored per angle bin] (nan for an empty bin, like the reference's mean of nothing)."""
        if not self.angle_bins:
            return []
        return [100.0 * h[2] / h[0] if h[0] else float("nan") for h in self.bin_hits.tolist()]

    def merge_(self, other_hits):
        self.hits += other_hits.to(self.hits.device)
        return self

    def summary(self):
        h = self.hits.tolist()
        tot = max(h[0], 1)
        mut = max(h[1], 1)
        n3, n2 = self.n3, self.n2
        return {
            "scored": h[0],
            "mutual": h[1],
            "recall_3d": {t: 100.0 * h[2 + i] / tot for i, t in enumerate(self.thr3d)},
            "recall_2d": {t: 100.0 * h[2 + n3 + i] / tot for i, t in enumerate(self.thr2d)},
            "mutual_recall_3d": {t: 100.0 * h[2 + n3 + n2 + i] / mut for i, t in enumerate(self.thr3d)},
            "mutual_recall_2d": {t: 100.0 * h[2 + 2 * n3 + n2 + i] / mut for i, t in enumerate(self.thr2d)},
        }


_SIDE_STREAMS = {}


def _both_sides(fn0, fn1, dev):
    """Prepare the two images of a pair concurrently: image 1 runs on a side stream forked from, and joined
    back into, the current stream (inside a CUDA-graph capture this becomes a fork / join in the graph), so
    its single-CTA compaction and small geometry kernels overlap image 0's work."""
    cur = torch.cuda.current_stream(dev)
    side = _SIDE_STREAMS.get(dev.index)
    if side is None:
        side = _SIDE_STREAMS[dev.index] = torch.cuda.Stream(device=dev)
    side.wait_stream(cur)
    s0 = fn0()
    with torch.cuda.stream(side):
        s1 = fn1()
    cur.wait_stream(side)
    for name in s1.__slots__:  # allocated on the side stream, consumed on the current one
        t = getattr(s1, name, None)
        if torch.is_tensor(t):
            t.record_stream(cur)
    return s0, s1


def match_and_score_depth(feat_0, feat_1, depth_0, depth_1, K, Rt, num_corr, acc, sync=False):
    """ScanNet-shaped pair, end to end on the device: estimate_correspondence_depth
    (correspondence.py:218-232) + the caller's error / recall block
    (render_scannet_correspondence.py:211-217, :253-264) with no host round trip when sync=False."""
    dev = C_._device()
    Kc = K.detach().float().cpu()
    Kh, Kinv = C_._host_mat(Kc), C_._host_mat(Kc.inverse())
    fm0, fm1, kw0, kw1 = C_._pair_maps(feat_0, feat_1, dev, depth_0.shape[-2] * depth_0.shape[-1], L.MV_SAMPLE_BILINEAR_ZEROS)
    s0, s1 = _both_sides(lambda: C_.prepare_depth_side(fm0, depth_0, Kh, Kinv, dev, sync=sync, **kw0),
                         lambda: C_.prepare_depth_side(fm1, depth_1, Kh, Kinv, dev, sync=sync, **kw1), dev)
    r = C_._match_sides(s0, s1, s0.n, s1.n, num_corr, n_dev=None if sync else s0.n_dev, m_dev=None if sync else s1.n_dev)
    acc.score(r, s0.xyz, s1.xyz, Rt, Kc)
    return r


def match_and_score_xyz(feat_0, feat_1, xyz_grid_0, xyz_grid_1, intrinsics, Rt, num_corr, acc, sync=False):
    """NAVI-shaped pair: estimate_correspondence_xyz (correspondence.py:235-263) + the caller's error /
    recall block (evaluate_navi_correspondence.py:186-212)."""
    dev = C_._device()
    fm0, fm1, kw0, kw1 = C_._pair_maps(feat_0, feat_1, dev, xyz_grid_0.shape[-2] * xyz_grid_0.shape[-1], L.MV_SAMPLE_BICUBIC_CLAMP)
    s0, s1 = _both_sides(lambda: C_.prepare_xyz_side(fm0, xyz_grid_0, dev, sync=sync, **kw0),
                         lambda: C_.prepare_xyz_side(fm1, xyz_grid_1, dev, sync=sync, **kw1), dev)
    r = C_._match_sides(s0, s1, s0.n, s1.n, num_corr, n_dev=None if sync else s0.n_dev, m_dev=None if sync else s1.n_dev)
    acc.score(r, s0.xyz, s1.xyz, Rt, intrinsics)
    return r


STAGE_MIN_BYTES = 1 << 15  # below this a plain copy_ is as fast; above, the driver's own pageable path also serialises with the stream


def copy_in(dst, src, stream=None):
    """dst.copy_(src) for a device tensor dst; a large PAGEABLE host tensor of the same dtype and memory order goes through
    the library's threaded pinned staging ring (mv_h2d_staged) instead of the driver's single-threaded staging."""
    if (src.device.type == "cpu" and not src.is_pinned() and src.dtype == dst.dtype and src.numel() == dst.numel()
            and src.numel() * src.element_size() >= STAGE_MIN_BYTES and src.stride() == dst.stride()
            and _dense(src) and _dense(dst)):
        st = stream if stream is not None else torch.cuda.current_stream(dst.device)
        L.call("mv_h2d_staged", c_void_p(dst.data_ptr()), c_void_p(src.data_ptr()), src.numel() * src.element_size(),
               c_void_p(st.cuda_stream))
        return
    dst.copy_(src, non_blocking=True)


def _dense(t):
    """True when the tensor's elements occupy one contiguous block (any permutation of a contiguous layout)."""
    if t.is_contiguous():
        return True
    order = sorted(range(t.dim()), key=lambda d: -t.stride(d))
    return t.permute(order).is_contiguous()


class GraphedPairMatcher:
    """The per-pair device pipeline (kernel 1 for both images, kernel 2, kernel 3 ratio / mutual / top-k)
    captured ONCE into a CUDA graph and replayed per pair: the ~25 launches of a pair cost one graph launch,
    so small pairs are no longer bound by host launch overhead.

    Shapes are fixed at construction; live point counts stay on the device (n_dev), so no host sync is
    needed between pairs.  Inputs are copied into static buffers (device -> device, or straight from
    pinned host memory), then `run()` replays the graph and scores the pair into a RecallAccumulator.

    kind = "xyz"   NAVI-shaped   : feats (C, h, w) x2 + xyz grids (3, H, W) x2
    kind = "depth" ScanNet-shaped: feats (C, h, w) x2 + depth (1, H, W) x2 + K (fixed for the matcher)
    """

    def __init__(self, kind, feat_shape, grid_shape, num_corr, K=None, device=None, ratio_test=True, with_outputs=False,
                 feat_layout="chw", feat_dtype=torch.float32, split=False, mutual=False):
        """feat_layout: memory layout of the static feature buffers -- "chw" (the reference's contiguous
        (C, h, w)) or "hwc" (channel-last views, the layout ViT tokens / channels_last CNN outputs already have:
        loading such features is a flat copy and the transpose kernel is skipped).
        mutual: select mutual matches with the two-sided ratio test (correspondence.get_mutual_correspondences) -- in the
        single graph and in the split form alike; the selection's length stays on the device (match.k_dev <= match.k), which
        RecallAccumulator.score reads there."""
        if kind not in ("xyz", "depth"):
            raise ValueError(kind)
        if not isinstance(mutual, bool):
            raise TypeError(f"mutual must be a bool, not {type(mutual).__name__}")
        self.mutual = mutual
        if feat_layout not in ("chw", "hwc"):
            raise ValueError(feat_layout)
        # split: TWO graphs -- the target image's side (its map, the f16c centre, kernel 1) and everything else -- so that a
        # host caller's upload of image 0 overlaps the target side's kernels (load_and_replay_split)
        self.split = bool(split)
        self.graph_target = None
        self.feat_layout = feat_layout
        self.feat_dtype = feat_dtype  # torch.bfloat16 / float16: 16-bit static buffers, widened on the device
        C_._check_C(feat_shape[0])
        self.kind, self.num_corr = kind, int(num_corr)
        self.ratio_test, self.with_outputs = bool(ratio_test), bool(with_outputs)
        self.packed = self.host_packed = None
        self.k_max = 0
        self.dev = device or C_._device()
        if feat_layout == "hwc":
            C, h, w = feat_shape
            self.f0 = torch.zeros((h, w, C), dtype=feat_dtype, device=self.dev).permute(2, 0, 1)
            self.f1 = torch.zeros((h, w, C), dtype=feat_dtype, device=self.dev).permute(2, 0, 1)
        else:
            self.f0 = torch.zeros(feat_shape, dtype=feat_dtype, device=self.dev)
            self.f1 = torch.zeros(feat_shape, dtype=feat_dtype, device=self.dev)
        self.g0 = torch.zeros(grid_shape, dtype=torch.float32, device=self.dev)
        self.g1 = torch.zeros(grid_shape, dtype=torch.float32, device=self.dev)
        if kind == "depth":
            # the intrinsics live in device memory ([K | K^-1], 18 floats) so that they can change between replays of
            # the captured graph (ScanNet's differ per scene); load(..., K=...) refreshes them
            self.Kdev = torch.zeros(18, dtype=torch.float32, device=self.dev)
            self.Kpin = torch.zeros((8, 18), dtype=torch.float32).pin_memory()  # ring of staging rows: no sync on a change
            self.Kevents = [None] * 8  # per row: recorded after the row's H2D copy; the row is rewritten only once it fired
            self.Kturn = 0
            self.Kc = None
            self.set_intrinsics(K)
        self.graph = None
        self.out = None

    def _prepare(self, fm, g, kw):
        if self.kind == "xyz":
            return C_.prepare_xyz_side(fm, g, self.dev, sync=False, **kw)
        Kd, Kinvd = L.ptr(self.Kdev), c_void_p(self.Kdev.data_ptr() + 36)
        return C_.prepare_depth_side(fm, g, Kd, Kinvd, self.dev, sync=False, **kw)

    def _exact(self):
        """the exact low-rank route (no kernel 1) for this matcher's shapes?"""
        C, h, w = self.f0.shape
        gp = self.g0.shape[-2] * self.g0.shape[-1]
        mode = L.MV_SAMPLE_BICUBIC_CLAMP if self.kind == "xyz" else L.MV_SAMPLE_BILINEAR_ZEROS
        return C_.lowrank_exact_applies(C, h, w, gp, gp, mode)

    def _body_target(self):
        """graph 1 of the split form: everything that needs only the TARGET image (image 1)."""
        fm1 = C_._feature_map(self.f1, self.dev)
        if self._exact():
            self._mu = None
            self._s1 = self._prepare(fm1, self.g1, {"want_rows": False})
            return
        f16 = C_._CFG["dtype"] != "bf16"  # f16c and tf32c rows are centred on the target
        self._mu = C_._center(fm1[0], fm1[0].shape[0], step=C_._center_step(fm1[0].shape[0])) if f16 else None
        kw1 = {"role": L.MV_ROLE_TARGET, "center": self._mu} if f16 else {}
        self._s1 = self._prepare(fm1, self.g1, kw1)

    def _body_query(self):
        """graph 2 of the split form: the query image's side, kernels 2 and 3, the packed outputs."""
        fm0 = C_._feature_map(self.f0, self.dev)
        kw0 = {"role": L.MV_ROLE_QUERY, "dotvec": self._mu, "pixdot": C_._rows_dot(fm0[0], self._mu)} if self._mu is not None else {}
        if self._exact():
            kw0 = {"want_rows": False}
        s0, s1 = self._prepare(fm0, self.g0, kw0), self._s1
        return self._match_and_pack(s0, s1)

    def _body(self):
        gp = self.g0.shape[-2] * self.g0.shape[-1]
        fm0, fm1, kw0, kw1 = C_._pair_maps(self.f0, self.f1, self.dev, gp,
                                           L.MV_SAMPLE_BICUBIC_CLAMP if self.kind == "xyz" else L.MV_SAMPLE_BILINEAR_ZEROS)
        if self.kind == "xyz":
            s0, s1 = _both_sides(lambda: C_.prepare_xyz_side(fm0, self.g0, self.dev, sync=False, **kw0),
                                 lambda: C_.prepare_xyz_side(fm1, self.g1, self.dev, sync=False, **kw1), self.dev)
        else:
            Kd, Kinvd = L.ptr(self.Kdev), c_void_p(self.Kdev.data_ptr() + 36)
            s0, s1 = _both_sides(lambda: C_.prepare_depth_side(fm0, self.g0, Kd, Kinvd, self.dev, sync=False, **kw0),
                                 lambda: C_.prepare_depth_side(fm1, self.g1, Kd, Kinvd, self.dev, sync=False, **kw1), self.dev)
        return self._match_and_pack(s0, s1)

    def _match_and_pack(self, s0, s1):
        self.lowrank_exact = s0.rows16 is None and s0.rows32 is None
        self.lowrank_used = (not self.lowrank_exact and s0.rows_lo is not None and s0.fshape == s1.fshape
                             and C_.lowrank_applies(*s0.fshape, s0.n, s1.n, s0.mode))
        r = C_._match_sides(s0, s1, s0.n, s1.n, self.num_corr, self.ratio_test, n_dev=s0.n_dev, m_dev=s1.n_dev, mutual=self.mutual)
        if self.with_outputs:
            # the helper's return tuple + the live counts in one buffer of column blocks (mv_pack_matches):
            # a single device -> host copy, and the host slices views out of it
            k = r.k
            self.k_max = k
            blocks = 11 if self.kind == "xyz" else 7
            self.packed = torch.empty(blocks * k + 4, dtype=torch.float32, device=self.dev)
            L.call("mv_pack_matches", L.ptr(r.sel_src), L.ptr(r.sel_dst), L.ptr(r.sel_weight), L.ptr(r.k_dev), k,
                   L.ptr(s0.xyz), L.ptr(s1.xyz), L.ptr(s0.uv) if self.kind == "xyz" else None,
                   L.ptr(s1.uv) if self.kind == "xyz" else None, L.ptr(s0.n_dev), L.ptr(s1.n_dev), L.ptr(self.packed),
                   C_._stream())
        return s0, s1, r

    def capture(self):
        """warm up (first-call attribute / entry-point initialisation must not happen under capture), then capture."""
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self._body()
        cur.wait_stream(side)
        torch.cuda.synchronize(self.dev)
        # torch.cuda.graph's default capture stream is created once per process on whatever device was current then: a
        # matcher on another device must bring its own, or its allocations fall outside the capture's pool
        cap = torch.cuda.Stream(device=self.dev)
        if self.split:
            pool = torch.cuda.graph_pool_handle()  # the second graph consumes tensors the first one produces
            self.graph_target = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_target, pool=pool, stream=cap):
                self._body_target()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, pool=pool, stream=cap):
                self.out = self._body_query()
        else:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=cap):
                self.out = self._body()
        if self.with_outputs:
            self.host_packed = torch.empty(self.packed.shape, dtype=torch.float32, pin_memory=True)
        return self

    def set_intrinsics(self, K):
        """(depth kind) K (3, 3) for the following replays; a no-op when it is the matrix already loaded."""
        Kc = K.detach().float().cpu().reshape(3, 3)
        if self.Kc is not None and torch.equal(Kc, self.Kc):
            return
        self.Kc = Kc.clone()
        slot = self.Kturn % 8
        self.Kturn += 1
        row = self.Kpin[slot]
        # the host may run many pairs ahead of the GPU (PairPipeline.submit never syncs): a queued copy from this row
        # could still be pending 8 changes later, so wait for ITS event before overwriting the staging memory
        ev = self.Kevents[slot]
        if ev is not None:
            ev.synchronize()
        row[:9] = Kc.reshape(-1)
        row[9:] = Kc.inverse().reshape(-1)
        self.Kdev.copy_(row, non_blocking=True)
        if ev is None:
            ev = self.Kevents[slot] = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))

    def load(self, feat_0, feat_1, grid_0, grid_1, two_streams=False, K=None):
        """stage one pair's inputs (any device; pinned host memory makes the copies asynchronous).
        K: (depth kind) the pair's intrinsics, if they differ from the ones the matcher was built with.
        two_streams: issue image 1's copies on a second stream -- two concurrent host -> device transfers use the
        PCIe link better than one (measured: 463 -> ~390 us for the 19.6 MB of a NAVI-shaped pair)."""
        if K is not None and self.kind == "depth":
            self.set_intrinsics(K)
        pageable = feat_0.device.type == "cpu" and not feat_0.is_pinned()
        if not two_streams or pageable:  # pageable sources: the staging threads already keep the link busy on one stream
            copy_in(self.f0, feat_0)
            copy_in(self.f1, feat_1)
            copy_in(self.g0, grid_0)
            copy_in(self.g1, grid_1)
            return
        cur = torch.cuda.current_stream(self.dev)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.dev)
        side = self._copy_stream
        side.wait_stream(cur)  # the static buffers may still be read by the previous replay
        with torch.cuda.stream(side):
            self.f1.copy_(feat_1, non_blocking=True)
            self.g1.copy_(grid_1, non_blocking=True)
        self.f0.copy_(feat_0, non_blocking=True)
        self.g0.copy_(grid_0, non_blocking=True)
        cur.wait_stream(side)

    def load_and_replay_split(self, feat_0, feat_1, grid_0, grid_1, K=None):
        """(split form, host tensors) upload the TARGET image first, replay its graph while the query image uploads, then
        replay the rest: the target side's ~60 us of kernels disappear behind the second half of the upload.  The copies go
        through one copy stream in order (image 1, then image 0), so image 1 owns the link until it is complete."""
        if K is not None and self.kind == "depth":
            self.set_intrinsics(K)
        cur = torch.cuda.current_stream(self.dev)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.dev)
            self._ev1, self._ev0 = torch.cuda.Event(), torch.cuda.Event()
        cp = self._copy_stream
        cp.wait_stream(cur)  # the static buffers may still be read by the previous replay
        with torch.cuda.stream(cp):
            copy_in(self.f1, feat_1, cp)
            copy_in(self.g1, grid_1, cp)
            self._ev1.record(cp)
        cur.wait_event(self._ev1)
        self.graph_target.replay()
        with torch.cuda.stream(cp):
            copy_in(self.f0, feat_0, cp)
            copy_in(self.g0, grid_0, cp)
            self._ev0.record(cp)
        cur.wait_event(self._ev0)
        self.graph.replay()
        L.LAUNCHES["count"] += self.launches_per_replay

    def run(self, acc=None, Rt=None, K=None):
        """replay the captured pipeline on the staged inputs; optionally score into `acc`."""
        if self.graph is None:
            self.capture()
        if self.graph_target is not None:
            self.graph_target.replay()
        self.graph.replay()
        L.LAUNCHES["count"] += self.launches_per_replay
        s0, s1, r = self.out
        if acc is not None:
            if K is None:
                if self.kind != "depth":
                    raise ValueError("run(acc=...) of an 'xyz' matcher needs the pair's intrinsics K (there is no matcher-wide K)")
                K = self.Kc
            acc.score(r, s0.xyz, s1.xyz, Rt, K)
        return r

    @property
    def launches_per_replay(self):
        # per image: (backproject) + compact + coords + chw_to_hwc + kernel 1; per pair: (centre: 2, pixel dots: 1) + kernel 2 (2) + ratio + top-k
        zero_copy = self.feat_layout == "hwc" and self.feat_dtype == torch.float32
        per_side = (5 if self.kind == "depth" else 4) - (1 if zero_copy else 0)
        # mutual: kernel 2's column merge, the reverse kernel 3, and the combine + count clamp around the top-k
        mutual = 4 if self.mutual else 0
        if getattr(self, "lowrank_exact", False):
            # per image everything but kernel 1; per pair: exact Gram (2), 2 builders, kernel 2 (2), kernel 3 on the Gram, top-k
            return 2 * (per_side - 1) + 8 + (1 if self.with_outputs else 0) + mutual
        lowrank = 6 if getattr(self, "lowrank_used", False) else 0  # 2 unit-row launches, the Gram launch + its row merge, 2 builders
        return 2 * per_side + 4 + (3 if C_._CFG["dtype"] != "bf16" else 0) + (1 if self.with_outputs else 0) + lowrank + mutual


class PairPipeline:
    """Several GraphedPairMatchers, each on its own stream, fed round-robin: while one pair sits in its
    low-occupancy phases (single-CTA compaction and top-k, the small geometry / ratio / scoring kernels) the
    next pair's kernel 1 / kernel 2 use the idle SMs.  All lanes accumulate into the same RecallAccumulator
    (device atomics), so the result is independent of the interleaving.

        pipe = PairPipeline("xyz", feat_shape, grid_shape, num_corr, lanes=2)
        for p in pairs: pipe.submit(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], acc, p["Rt"], p["intrinsics"])
        pipe.join()
    """

    def __init__(self, kind, feat_shape, grid_shape, num_corr, K=None, device=None, lanes=2, feat_layout="chw",
                 feat_dtype=torch.float32):
        self.dev = device or C_._device()
        self.lanes = []
        for _ in range(max(1, int(lanes))):
            st = torch.cuda.Stream(device=self.dev)
            with torch.cuda.stream(st):
                gm = GraphedPairMatcher(kind, feat_shape, grid_shape, num_corr, K=K, device=self.dev,
                                        feat_layout=feat_layout, feat_dtype=feat_dtype).capture()
            self.lanes.append((st, gm))
        torch.cuda.synchronize(self.dev)
        self.turn = 0

    def submit(self, feat_0, feat_1, grid_0, grid_1, acc=None, Rt=None, K=None):
        st, gm = self.lanes[self.turn % len(self.lanes)]
        self.turn += 1
        st.wait_stream(torch.cuda.current_stream(self.dev))  # inputs produced on the caller's stream
        with torch.cuda.stream(st):
            gm.load(feat_0, feat_1, grid_0, grid_1, K=K if gm.kind == "depth" else None)
            return gm.run(acc, Rt, K)

    def join(self):
        """make the caller's stream wait for every lane (call before reading the accumulator)."""
        cur = torch.cuda.current_stream(self.dev)
        for st, _ in self.lanes:
            cur.wait_stream(st)
