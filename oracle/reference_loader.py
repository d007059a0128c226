"""TEST INFRASTRUCTURE ONLY.  Import the reference's own matching code, unmodified, from a checkout of the
reference project: $MV_REFERENCE_ROOT, or oracle/_ref/ (git-ignored; the reference is not part of this repository).

Callers must check `available()` first.  Used by oracle/make_golden.py and by the CPU tests that pin
oracle/restated.py to the real thing (tests/test_oracle.py, which falls back to stored values without it).
"""
import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get("MV_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "evals", "utils", "correspondence.py"))


def load():
    """-> (evals.utils.correspondence, evals.utils.transformations) of the reference."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    from . import faiss_shim

    faiss_shim.install()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    corr = importlib.import_module("evals.utils.correspondence")
    tr = importlib.import_module("evals.utils.transformations")
    return corr, tr


def load_spair():
    """-> the reference's own `compute_errors` / `evaluate_dataset` (evaluate_spair_correspondence.py:45-123),
    unmodified.  The script imports hydra / omegaconf (not installed here) only for its `main`; both are
    replaced by empty stand-ins.  `compute_errors` moves tensors with `.cuda()`, which has no meaning in the
    GPU-less build container: use `spair_compute_errors_reference`, which maps `.cuda()` to the identity
    for the duration of the call."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    import types

    if "hydra" not in sys.modules:
        hydra = types.ModuleType("hydra")
        hydra.main = lambda *a, **k: (lambda fn: fn)
        hydra_utils = types.ModuleType("hydra.utils")
        hydra_utils.instantiate = lambda *a, **k: None
        hydra.utils = hydra_utils
        sys.modules["hydra"], sys.modules["hydra.utils"] = hydra, hydra_utils
    if "omegaconf" not in sys.modules:
        oc = types.ModuleType("omegaconf")
        oc.DictConfig, oc.OmegaConf = dict, type("OmegaConf", (), {})
        sys.modules["omegaconf"] = oc
    from . import faiss_shim

    faiss_shim.install()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    return importlib.import_module("evaluate_spair_correspondence")


def spair_compute_errors_reference(feats, kps_i, kps_j, thresh_scale, image_size):
    """run the reference's compute_errors on given backbone features: the `model` is a stand-in that returns
    `feats`, the images / masks are blanks of the right size (masks are only used with mask_feats=True)."""
    import numpy as np
    import torch

    mod = load_spair()
    img = torch.zeros(3, image_size, image_size)
    mask = np.ones((image_size, image_size), dtype=float)
    instance = (img, mask, kps_i.clone(), img, mask, kps_j.clone(), thresh_scale, None)
    real_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        return mod.compute_errors(lambda images: feats.clone(), instance, return_heatmaps=True)
    finally:
        torch.Tensor.cuda = real_cuda


def spair_evaluate_dataset_reference(pairs, thresh=0.10):
    """the reference's evaluate_dataset (evaluate_spair_correspondence.py:106-123) over a list of synthetic pairs
    (dicts with feats, kps_i, kps_j, thresh_scale, image_size): -> (recall, confusion)."""
    import numpy as np
    import torch

    mod = load_spair()
    calls = {"i": 0}

    class Data:
        def __len__(self):
            return len(pairs)

        def __getitem__(self, i):
            p = pairs[i]
            calls["i"] = i
            img = torch.zeros(3, p["image_size"], p["image_size"])
            mask = np.ones((p["image_size"], p["image_size"]), dtype=float)
            return (img, mask, p["kps_i"].clone(), img, mask, p["kps_j"].clone(), p["thresh_scale"], None)

    real_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        return mod.evaluate_dataset(lambda images: pairs[calls["i"]]["feats"].clone(), Data(), thresh)
    finally:
        torch.Tensor.cuda = real_cuda


def navi_error_block_reference(feats_0, feats_1, xyz_grid_0, xyz_grid_1, Rt_gt, intrinsics, num_corr, scale_factor=0.25):
    """Execute the reference's OWN NAVI evaluation loop -- the text of evaluate_navi_correspondence.py from
    `num_instances = len(loader.dataset)` up to the CSV header (lines 174-221), read from REFERENCE_ROOT at call time,
    never copied into this repo -- with the script's names bound to the reference's own functions (faiss shimmed),
    tqdm / wandb / print silenced and cfg / loader replaced by stand-ins.  Returns the variables the block leaves
    behind."""
    import types

    import numpy as np
    import torch

    corr, tr = load()
    path = os.path.join(REFERENCE_ROOT, "evaluate_navi_correspondence.py")
    lines = open(path).read().splitlines()
    beg = next(i for i, l in enumerate(lines) if "num_instances = len(loader.dataset)" in l)
    end = next(i for i, l in enumerate(lines) if "# Define the header for the CSV file" in l)
    import textwrap

    block = textwrap.dedent("\n".join(lines[beg:end]))
    ns = {
        "torch": torch, "np": np, "tqdm": lambda it: it, "print": lambda *a, **k: None,
        "wandb": types.SimpleNamespace(log=lambda *a, **k: None),
        "cfg": types.SimpleNamespace(num_corr=num_corr, scale_factor=scale_factor),
        "loader": types.SimpleNamespace(dataset=list(range(len(feats_0)))),
        "estimate_correspondence_xyz": corr.estimate_correspondence_xyz, "project_3dto2d": corr.project_3dto2d,
        "compute_binned_performance": corr.compute_binned_performance, "transform_points_Rt": tr.transform_points_Rt,
        "so3_rotation_angle": tr.so3_rotation_angle,
        "feats_0": feats_0, "feats_1": feats_1, "xyz_grid_0": xyz_grid_0, "xyz_grid_1": xyz_grid_1, "Rt_gt": Rt_gt,
        "intrinsics": intrinsics,
    }
    exec(compile(block, path, "exec"), ns)  # noqa: S102 -- the reference's own text, test infrastructure only
    return {"err_3d": ns["err_3d"], "err_2d": ns["err_2d"], "results": ns["results"], "bin_rec": ns["bin_rec"],
            "rec_2cm": ns["rec_2cm"], "rel_ang": ns["rel_ang"]}


def _exec_lines(path, first_marker, last_marker, ns):
    """exec the lines of a reference file from the one containing first_marker to the one containing last_marker."""
    import textwrap

    lines = open(os.path.join(REFERENCE_ROOT, path)).read().splitlines()
    beg = next(i for i, l in enumerate(lines) if first_marker in l)
    end = next(i for i, l in enumerate(lines) if last_marker in l and i >= beg)
    exec(compile(textwrap.dedent("\n".join(lines[beg:end + 1])), path, "exec"), ns)  # noqa: S102 -- the reference's own text
    return ns


def maskcut_affinity_reference(feats, tau, eps=1e-5):
    """the reference's own affinity lines (evals/models/maskcut_processor.py:77-78 and :103-106), executed from its file
    (the module itself needs pydensecrf / sklearn / wandb to import): -> (A_raw, A_thresholded, d_i)."""
    import numpy as np
    import torch.nn.functional as F

    ns = {"feats": feats, "F": F, "np": np}
    _exec_lines("evals/models/maskcut_processor.py", "feats = F.normalize(feats, p=2, dim=0)", "A = (feats.transpose(0, 1) @ feats).cpu().numpy()", ns)
    raw = ns["A"].copy()
    ns.update({"tau": tau, "eps": eps})
    _exec_lines("evals/models/maskcut_processor.py", "A = A > tau", "d_i = np.sum(A, axis=1)", ns)
    return raw, ns["A"], ns["d_i"]


def twoafc_reference(ref, left, right):
    """cosine_similarity_batch of evaluate_model_percepture.py:46-48 and the prediction line :120-122, from the file."""
    import torch
    import torch.nn.functional as F

    ns = {"F": F, "torch": torch}
    _exec_lines("evaluate_model_percepture.py", "def cosine_similarity_batch(tensor1, tensor2):", "return F.cosine_similarity(tensor1, tensor2, dim=-1)", ns)
    ns.update({"features_ref": ref, "features_left": left, "features_right": right})
    ns["similarity_left"] = ns["cosine_similarity_batch"](ref, left)
    ns["similarity_right"] = ns["cosine_similarity_batch"](ref, right)
    _exec_lines("evaluate_model_percepture.py", "predictions = torch.where(similarity_left > similarity_right, 0, 1)",
                "predictions = torch.where(similarity_left > similarity_right, 0, 1)", ns)
    return ns["similarity_left"], ns["similarity_right"], ns["predictions"]
