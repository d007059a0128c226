"""TEST INFRASTRUCTURE ONLY.  Generate tests/golden/*.npz by running the reference's OWN module
(evals/utils/correspondence.py of a checkout of the reference project at oracle/_ref/ or
$MV_REFERENCE_ROOT, imported unmodified through oracle/reference_loader.py
with the exact brute-force faiss stand-in) on the seeded synthetic inputs of
midvision-probe_b200/synthetic.py.  Needs that checkout:

    python -m oracle.make_golden

The SPair case has no importable reference (its matching is inlined in a Hydra script that needs
hydra + a CUDA device), so its fixture is produced by oracle/restated.py and is marked as such.
"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden")

# small shapes: the whole set is a few hundred kB
SCANNET_SMALL = dict(C=64, h=6, w=8, H=24, W=32)
NAVI_SMALL = dict(C=64, h=8, w=8, H=32, W=32, radius=12.0)
SPAIR_SMALL = dict(C=64, h=14, w=14, K=20, image_size=224)
ROWS_SMALL = dict(n=300, m=280, C=64)


def np32(t):
    return t.detach().cpu().numpy()


def main():
    from oracle import reference_loader, restated

    syn = importlib.import_module("midvision-probe_b200.synthetic")
    ref, ref_tr = reference_loader.load()
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)  # summation order of the fixture is then machine independent

    for coherent in (True, False):
        tag = "coh" if coherent else "rnd"
        p = syn.scannet_pair(7, coherent=coherent, **SCANNET_SMALL)
        x0, x1, w = ref.estimate_correspondence_depth(p["feat_0"], p["feat_1"], p["depth_0"], p["depth_1"], p["K"].clone(), 100)
        Kinv = p["K"].inverse()
        pc = ref.grid_to_pointcloud(Kinv, p["depth_0"])
        pc_valid = pc[pc[:, 2] > 0]
        pcF = ref.sample_pointcloud_features(p["feat_0"], p["K"].clone(), pc_valid, p["depth_0"].shape[-2:])
        e3 = (ref_tr.transform_points_Rt(x0, p["Rt"]) - x1).norm(p=2, dim=1)
        np.savez_compressed(os.path.join(OUT, f"scannet_small_{tag}.npz"), source="reference", index=7,
                            feat_checksum=np32(p["feat_0"].double().sum()), corr_xyz0=np32(x0), corr_xyz1=np32(x1),
                            corr_dist=np32(w), pointcloud=np32(pc), sampled=np32(pcF), err3d=np32(e3))

        p = syn.navi_pair(7, coherent=coherent, **NAVI_SMALL)
        out = ref.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 100)
        out_nr = ref.estimate_correspondence_xyz(p["feat_0"], p["feat_1"], p["xyz_grid_0"], p["xyz_grid_1"], 100, ratio_test=False)
        np.savez_compressed(os.path.join(OUT, f"navi_small_{tag}.npz"), source="reference", index=7,
                            feat_checksum=np32(p["feat_0"].double().sum()), c_xyz0=np32(out[0]), c_xyz1=np32(out[1]),
                            c_dist=np32(out[2]), c_uv0=np32(out[3]), c_uv1=np32(out[4]), nr_dist=np32(out_nr[2]),
                            nr_xyz0=np32(out_nr[0]))

    g = torch.Generator().manual_seed(4242)
    X = torch.randn(ROWS_SMALL["n"], ROWS_SMALL["C"], generator=g)
    Y = torch.randn(ROWS_SMALL["m"], ROWS_SMALL["C"], generator=g)
    d, i = ref.knn_points(X, Y, 2, "cosine")
    i1, i2, w = ref.get_correspondences_ratio_test(X, Y, 50)
    rt = ref.calculate_ratio_test(d)
    hm = torch.randn(5, 7, 9, generator=g)
    uv = ref.project_3dto2d(torch.randn(11, 3, generator=g) + torch.tensor([0.0, 0.0, 3.0]), torch.tensor([[500.0, 0, 320], [0, 500, 240], [0, 0, 1]]))
    np.savez_compressed(os.path.join(OUT, "rows_small.npz"), source="reference", seed=4242, dists=np32(d), idx=np32(i),
                        idx1=np32(i1), idx2=np32(i2), weight=np32(w), ratio=np32(rt), heat=np32(hm),
                        argmax=np32(ref.argmax_2d(hm)), argmin=np32(ref.argmax_2d(hm, max_value=False)),
                        grid=np32(ref.get_grid(3, 5)), uv=np32(uv))

    p = syn.spair_pair(7, **SPAIR_SMALL)
    # the reference's own compute_errors (evaluate_spair_correspondence.py:45-103), hydra / omegaconf stubbed and
    # .cuda() mapped to the identity (oracle/reference_loader.py)
    es, en, isame, inn, heat = reference_loader.spair_compute_errors_reference(p["feats"], p["kps_i"], p["kps_j"], p["thresh_scale"], p["image_size"])
    np.savez_compressed(os.path.join(OUT, "spair_small.npz"), source="reference",
                        index=7, error_same=np32(es), error_nn=np32(en), index_same=np32(isame), index_nn=np32(inn),
                        pred=np32(restated.argmax_2d(heat)))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
