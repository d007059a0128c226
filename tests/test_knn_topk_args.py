"""Argument checks of the k > 2 nearest-neighbour entry points (kernel 2's top-KP epilogue, the fp32 re-rank): reported
through the status code + mv_last_error() before any CUDA call, so they run without a GPU."""
import ctypes


def test_topk_entry_points_validate_before_touching_cuda(mv):
    lib = mv.load()
    P16 = ctypes.c_void_p(16)
    E_ARG, E_RANGE, E_WORKSPACE = -1, -3, -4
    ws_big = ctypes.c_size_t(1 << 30)

    def topk(A=P16, kp=8, ws=P16, ws_bytes=ws_big, row_idx=P16):
        return lib.mv_k2_sim_topk_ld(A, 64, P16, 64, 1000, 1000, 64, None, None, 0, 0, kp, P16, row_idx, ws, ws_bytes, None)

    def rerank(Q=P16, cand=P16, kp=8, k=3, metric=0):
        return lib.mv_knn_rerank(Q, 64, P16, 64, 64, None, 100, cand, kp, k, metric, P16, P16, None)

    cases = [
        ("mv_k2_sim_topk_ld", lambda: topk(A=None), E_ARG),
        ("mv_k2_sim_topk_ld", lambda: topk(row_idx=None), E_ARG),
        ("mv_k2_sim_topk_ld", lambda: topk(ws=None), E_ARG),
        ("mv_k2_sim_topk_ld", lambda: topk(kp=4), E_RANGE),
        ("mv_k2_sim_topk_ld", lambda: topk(kp=32), E_RANGE),
        ("mv_k2_sim_topk_ld", lambda: topk(ws_bytes=ctypes.c_size_t(1024)), E_WORKSPACE),
        ("mv_knn_rerank", lambda: rerank(Q=None), E_ARG),
        ("mv_knn_rerank", lambda: rerank(cand=None), E_ARG),
        ("mv_knn_rerank", lambda: rerank(kp=4, k=3), E_RANGE),
        ("mv_knn_rerank", lambda: rerank(kp=8, k=9), E_RANGE),
        ("mv_knn_rerank", lambda: rerank(kp=8, k=0), E_RANGE),
        ("mv_knn_rerank", lambda: rerank(metric=2), E_ARG),
    ]
    for name, call, want in cases:
        rc = call()
        assert rc == want, f"{name}: rc={rc}, wanted {want}: {lib.mv_last_error()}"
        assert name.encode() in lib.mv_last_error()


def test_topk_workspace_size(mv):
    lib = mv.load()
    assert lib.mv_k2_topk_workspace_bytes(1000, 1000, 4) == 0  # not a list length
    w8, w16 = lib.mv_k2_topk_workspace_bytes(1000, 1000, 8), lib.mv_k2_topk_workspace_bytes(1000, 1000, 16)
    assert 0 < w8 <= w16 and w8 % 256 == 0 and w16 % 256 == 0
    assert lib.mv_k2_topk_workspace_bytes(20000, 1000, 16) > w16
