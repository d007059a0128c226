"""Argument checks of the mutual-matching entry points: the C ABI reports them through the status code +
mv_last_error() before any CUDA call, and the Python keywords are checked before any device work, so all of this runs
without a GPU."""
import ctypes

import pytest
import torch


def test_mutual_entry_points_validate_before_touching_cuda(mv):
    lib = mv.load()
    P16 = ctypes.c_void_p(16)
    E_ARG, E_ALIGN, E_RANGE, E_WORKSPACE = -1, -2, -3, -4
    ws_big = ctypes.c_size_t(1 << 34)

    def cols(A=P16, C=64, col_idx=P16, col_val=P16, ws=P16, ws_bytes=ws_big, dtype=0, n=1000):
        return lib.mv_k2_sim_top2_cols_ld(A, 64, P16, 64, n, 1000, C, None, None, dtype, 0, P16, P16, col_val, col_idx, P16, ws,
                                          ws_bytes, None)

    def select(row_idx=P16, k_dev=P16, n=100, num_corr=10):
        return lib.mv_k3_mutual_select(row_idx, P16, P16, P16, None, n, 1, num_corr, P16, None, P16, P16, P16, k_dev, None)

    def f16c_ab(A_hi=P16, center_A=P16, pitch=72, C=64):
        return lib.mv_k3_ratio_mutual_f16c_ab(A_hi, P16, P16, P16, C, pitch, center_A, None, None, 10, P16, None, 1, None, P16,
                                              None, None)

    cases = [
        ("mv_k2_sim_top2_cols_ld", lambda: cols(A=None), E_ARG),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(col_idx=None), E_ARG),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(col_val=None), E_ARG),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(ws=None), E_ARG),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(C=60), E_ALIGN),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(dtype=7), E_ARG),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(n=0), E_ARG),
        ("mv_k2_sim_top2_cols_ld", lambda: cols(ws_bytes=ctypes.c_size_t(1024)), E_WORKSPACE),
        ("mv_k3_mutual_select", lambda: select(row_idx=None), E_ARG),
        ("mv_k3_mutual_select", lambda: select(k_dev=None), E_ARG),
        ("mv_k3_mutual_select", lambda: select(n=-1), E_RANGE),
        ("mv_k3_mutual_select", lambda: select(num_corr=20000), E_RANGE),
        ("mv_k3_ratio_mutual_f16c_ab", lambda: f16c_ab(A_hi=None), E_ARG),
        ("mv_k3_ratio_mutual_f16c_ab", lambda: f16c_ab(center_A=ctypes.c_void_p(20)), E_ALIGN),
        ("mv_k3_ratio_mutual_f16c_ab", lambda: f16c_ab(pitch=64), E_ARG),
        ("mv_k3_ratio_mutual_f16c_ab", lambda: f16c_ab(C=60), E_ALIGN),
    ]
    for name, call, want in cases:
        rc = call()
        assert rc == want, f"{name}: rc={rc}, wanted {want}: {lib.mv_last_error()}"
        assert name.encode() in lib.mv_last_error()


def test_cols_workspace_size(mv):
    lib = mv.load()
    assert lib.mv_k2_cols_workspace_bytes(0, 1000) == 0 and lib.mv_k2_cols_workspace_bytes(1000, 0) == 0
    rows = lib.mv_k2_workspace_bytes(5024, 5024)
    w = lib.mv_k2_cols_workspace_bytes(5024, 5024)
    # one 16-byte record per (128-row block, column) behind the row records: 3.2 MB at 5024^2
    assert w - 40 * 5024 * 16 > 0 and w - 40 * 5024 * 16 <= rows
    assert lib.mv_k2_cols_workspace_bytes(18231, 18231) >= 143 * 18231 * 16


def test_mutual_keywords_are_checked_first(mv):
    C_ = mv.correspondence
    P = torch.zeros(10, 64)
    with pytest.raises(TypeError):
        C_.get_mutual_correspondences(P, P, 5, ratio_test=1)
    with pytest.raises(ValueError):
        C_.get_mutual_correspondences(P, P, -1)
    with pytest.raises(ValueError):
        C_.get_mutual_correspondences(P, P, 5.0)
    with pytest.raises(ValueError, match="multiple of 8"):
        C_.get_mutual_correspondences(torch.zeros(10, 60), torch.zeros(10, 60), 5)
    with pytest.raises(ValueError):
        C_.get_mutual_correspondences(torch.zeros(10, 64), torch.zeros(10, 72), 5)
    with pytest.raises(ValueError, match="too few"):
        C_.get_mutual_correspondences(torch.zeros(1, 64), P, 5)
    f, g = torch.zeros(64, 4, 4), torch.zeros(3, 8, 8)
    for bad in (1, "yes", None):
        with pytest.raises(TypeError):
            C_.estimate_correspondence_xyz(f, f, g, g, 10, mutual=bad)
        with pytest.raises(TypeError):
            C_.estimate_correspondence_depth(f, f, g[:1], g[:1], torch.eye(3), 10, mutual=bad)
    ev = mv.evaluation
    with pytest.raises(TypeError):
        ev.GraphedPairMatcher("xyz", (64, 4, 4), (3, 8, 8), 10, mutual=1)
