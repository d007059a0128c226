"""Argument checks of mv_spair_match_batch_tiled and its workspace query: reported through the status code +
mv_last_error() before any CUDA call, so they run without a GPU."""
import ctypes

MV_FEAT_F32, MV_FEAT_BF16, MV_FEAT_F16 = 0, 1, 2
E_ARG, E_ALIGN, E_RANGE, E_WORKSPACE = -1, -2, -3, -4


def test_workspace_query(mv):
    lib = mv.load()
    q = lib.mv_spair_tiled_workspace_bytes
    big = q(16, 768, 50, 50, 30)
    assert big > 0
    # slots + tap-norm partials + key-point fragments: grows with B, C and K, not with the map size
    assert q(32, 768, 50, 50, 30) > big and q(16, 2048, 50, 50, 30) > big and q(16, 768, 50, 50, 64) > big
    assert q(16, 768, 57, 57, 30) == big
    # bad sizes -> 0; no work -> 0
    for args in [(-1, 768, 50, 50, 30), (16, 0, 50, 50, 30), (16, 768, 0, 50, 30), (16, 768, 50, -2, 30),
                 (16, 768, 50, 50, 65), (16, 768, 50, 50, -1), (16, 768, 1025, 1025, 30), (0, 768, 50, 50, 30),
                 (16, 768, 50, 50, 0)]:
        assert q(*args) == 0, args


def test_tiled_validates_before_touching_cuda(mv):
    lib = mv.load()
    P16 = ctypes.c_void_p(16)
    f = ctypes.c_float
    need = lib.mv_spair_tiled_workspace_bytes(2, 64, 20, 20, 4)

    def tiled(feats=P16, dtype=MV_FEAT_F32, B=2, C=64, h=20, w=20, K=4, ws=P16, ws_bytes=None, confusion=None, conf_dim=0):
        return lib.mv_spair_match_batch_tiled(feats, dtype, B, C, h, w, P16, P16, K, 3, P16, f(320.0), f(0.1), None, None,
                                              None, None, None, confusion, conf_dim, ws,
                                              ctypes.c_size_t(need if ws_bytes is None else ws_bytes), None)

    cases = [
        (lambda: tiled(ws=None), E_WORKSPACE),                            # missing workspace
        (lambda: tiled(ws_bytes=need - 1), E_WORKSPACE),                  # one byte short
        (lambda: tiled(ws_bytes=0), E_WORKSPACE),
        (lambda: tiled(dtype=MV_FEAT_BF16, ws=None), E_WORKSPACE),
        (lambda: tiled(dtype=3), E_ARG),                                  # not an MV_FEAT_* value
        (lambda: tiled(dtype=-1, B=0), E_ARG),                            # a bad dtype is an error even without work
        (lambda: tiled(feats=None), E_ARG),
        (lambda: tiled(feats=ctypes.c_void_p(17), dtype=MV_FEAT_BF16), E_ALIGN),
        (lambda: tiled(feats=ctypes.c_void_p(18), dtype=MV_FEAT_F32), E_ALIGN),
        (lambda: tiled(K=65), E_RANGE),
        (lambda: tiled(h=1025, w=1025), E_RANGE),
        (lambda: tiled(confusion=P16, conf_dim=3), E_ARG),                # conf_dim < K
    ]
    for call, want in cases:
        rc = call()
        assert rc == want, f"rc={rc}, wanted {want}: {lib.mv_last_error()}"
        assert b"mv_spair_match_batch_tiled" in lib.mv_last_error()
    # no work: nothing is needed, whatever the (valid) element type
    for dtype in (MV_FEAT_F32, MV_FEAT_BF16, MV_FEAT_F16):
        assert tiled(feats=None, dtype=dtype, B=0, ws=None, ws_bytes=0) == 0
        assert tiled(feats=None, dtype=dtype, K=0, ws=None, ws_bytes=0) == 0
