"""Kernel 1's C = 3072 bicubic f16c rows, which leave through bulk stores (csrc/k1_sample.cu, BULK form), against the
per-row code of the MVMATCH_K1_WIDE=1 form: the hi plane (augmentation columns and untouched padding included), the lo
plane and row_dot must be the same bits.  The switch is read once per process, so each form runs in a process of its own
over the same saved inputs; the default form runs every case twice (repeatability)."""
import importlib
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C, h, w, H, W = 3072, 28, 28, 112, 112
SENTINEL = 0x5A5A  # every output element starts as this pattern: what a form does not write must stay so

# runs in a fresh interpreter: argv = inputs file, outputs file, launches per case
WORKER = r"""
import importlib, sys
import torch
mv = importlib.import_module("midvision-probe_b200")
L = mv._lib
inp = torch.load(sys.argv[1])
reps = int(sys.argv[3])
S = 0x5A5A
out = {}
for name, cs in inp["cases"].items():
    src = inp["maps"][cs["map"]].cuda()
    coords = inp["coords"][cs["map"]][: cs["n_max"]].cuda()
    n_max = cs["n_max"]
    n_dev = torch.tensor([cs["n_live"]], dtype=torch.int32, device="cuda") if cs["n_live"] is not None else None
    mu = inp["mu"][cs["map"]].cuda()
    center = mu if cs["center"] else None
    dotvec = mu if cs["dotvec"] else None
    pixdot = None
    if cs["pixdot"]:
        pixdot = torch.empty(src.shape[0], dtype=torch.float32, device="cuda")
        L.call("mv_rows_dot", L.ptr(src), src.shape[1], src.shape[0], L.ptr(mu), L.ptr(pixdot), None)
    runs = []
    for _ in range(reps):
        hi = torch.full((n_max, L.f16c_pitch(src.shape[1])), S, dtype=torch.int16, device="cuda")
        lo = torch.full((n_max, src.shape[1]), S, dtype=torch.int16, device="cuda")
        rd = torch.full((n_max,), S, dtype=torch.int32, device="cuda")
        L.call("mv_k1_sample_f16c", L.MV_SAMPLE_BICUBIC_CLAMP, L.ptr(src), src.shape[1], inp["h"], inp["w"], L.ptr(coords),
               L.ptr(n_dev), n_max, 1, cs["role"], L.ptr(center), L.ptr(dotvec), L.ptr(pixdot), L.ptr(hi), hi.shape[1], L.ptr(lo),
               None, L.ptr(rd), None, None)
        torch.cuda.synchronize()
        runs.append((hi.cpu(), lo.cpu(), rd.cpu()))
    out[name] = runs
torch.save(out, sys.argv[2])
"""


def _live_coords(xyz_grid):
    """bicubic source coordinates of the live (z > 0) pixels of the H x W grid, row-major: scale * (dst + 0.5) - 0.5 in
    fp32 (exact here: the scale is 1/4), as mv_geom_grid_coords computes them."""
    p = (xyz_grid[2].reshape(-1) > 0).nonzero().squeeze(1)
    x, y = (p % W).float(), (p // W).float()
    return torch.stack((0.25 * (x + 0.5) - 0.5, 0.25 * (y + 0.5) - 0.5), dim=1).contiguous()


def _mean_direction(src):
    return torch.nn.functional.normalize(src, dim=1).mean(0).contiguous()


Q, T = 0, 1  # MV_ROLE_QUERY, MV_ROLE_TARGET (include/mvmatch.h)
# name -> (map, role, centre, dotvec, pixdot, n_max, live count read on the device); n_max None = every live pixel,
# negative = that many fewer
CASES = {}
for _m in ("gauss0", "gauss1", "vit"):
    CASES[f"{_m}_query_pixdot"] = (_m, Q, False, False, True, None, None)  # the pipeline's query side
    CASES[f"{_m}_target_center"] = (_m, T, True, False, False, None, None)  # the pipeline's target side
    CASES[f"{_m}_query_center_dotvec"] = (_m, Q, True, True, False, None, None)
    CASES[f"{_m}_target_plain"] = (_m, T, False, False, False, None, None)
for _n in (-1, 148 * 30 + 1, 1000, 147, 100, 13, 1):  # short last ranges, fewer points than CTAs
    CASES[f"gauss0_query_n{_n}" if _n > 0 else f"gauss0_query_all_but{-_n}"] = ("gauss0", Q, False, False, True, _n, None)
CASES["gauss0_target_ndev"] = ("gauss0", T, True, False, False, None, 1675)


@pytest.fixture(scope="module")
def planes(tmp_path_factory):
    syn = importlib.import_module("midvision-probe_b200.synthetic")
    bb = importlib.import_module("midvision-probe_b200.backbones")
    maps, coords = {}, {}
    for i in (0, 1):
        g = torch.Generator().manual_seed(100 + i)
        maps[f"gauss{i}"] = torch.randn(h * w, C, generator=g)
        coords[f"gauss{i}"] = _live_coords(syn.navi_pair(i, C=8)["xyz_grid_0"])
    p = bb.navi_backbone_pair(0, device="cuda", noise=0.7)
    maps["vit"] = p["feat_0"].cpu().reshape(C, h * w).t().contiguous()
    coords["vit"] = _live_coords(p["xyz_grid_0"])
    mu = {k: _mean_direction(m) for k, m in maps.items()}
    cases = {}
    for name, (m, role, center, dotvec, pixdot, n_max, n_live) in CASES.items():
        n_all = coords[m].shape[0]
        n_max = n_all if n_max is None else (n_all + n_max if n_max < 0 else n_max)
        assert n_live is None or n_live < n_max
        cases[name] = dict(map=m, role=role, center=center, dotvec=dotvec, pixdot=pixdot, n_max=n_max, n_live=n_live)
    tmp = tmp_path_factory.mktemp("k1_bulk")
    inp = os.path.join(tmp, "inputs.pt")
    torch.save({"maps": maps, "coords": coords, "mu": mu, "cases": cases, "h": h, "w": w}, inp)
    res = {"cases": cases}
    for form, wide, reps in (("bulk", "0", 2), ("wide", "1", 1)):
        outp = os.path.join(tmp, f"{form}.pt")
        env = dict(os.environ, MVMATCH_K1_WIDE=wide)
        r = subprocess.run([sys.executable, "-c", WORKER, inp, outp, str(reps)], cwd=ROOT, env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-4000:]
        res[form] = torch.load(outp)
    return res


@pytest.mark.parametrize("name", list(CASES))
def test_bulk_rows_match_wide_form_bit_for_bit(planes, name):
    (hi, lo, rd), = planes["wide"][name]
    bhi, blo, brd = planes["bulk"][name][0]
    cs = planes["cases"][name]
    n = cs["n_live"] if cs["n_live"] is not None else cs["n_max"]
    assert torch.equal(bhi, hi) and torch.equal(blo, lo) and torch.equal(brd, rd)
    # every live row was written; the hi padding columns and the rows beyond the live count were not
    assert not (hi[:n, : C + 8] == SENTINEL).all(dim=1).any() and not (lo[:n] == SENTINEL).all(dim=1).any()
    assert (hi[:, C + 8:] == SENTINEL).all() and (hi[n:] == SENTINEL).all() and (lo[n:] == SENTINEL).all()
    assert (rd[:n] != SENTINEL).all() and (rd[n:] == SENTINEL).all()


@pytest.mark.parametrize("name", ["gauss0_query_pixdot", "vit_target_center", "gauss0_query_n13"])
def test_bulk_rows_repeat(planes, name):
    a, b = planes["bulk"][name]
    assert all(torch.equal(x, y) for x, y in zip(a, b))
