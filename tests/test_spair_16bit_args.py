"""Argument checks of mv_spair_match_batch_typed, the SPair batch entry point for fp32 / bf16 / fp16 maps: reported through
the status code + mv_last_error() before any CUDA call, so they run without a GPU."""
import ctypes

MV_FEAT_F32, MV_FEAT_BF16, MV_FEAT_F16 = 0, 1, 2


def test_spair_typed_validates_before_touching_cuda(mv):
    lib = mv.load()
    P16 = ctypes.c_void_p(16)
    E_ARG, E_ALIGN, E_RANGE = -1, -2, -3
    f = ctypes.c_float

    def typed(feats=P16, dtype=MV_FEAT_BF16, B=2, K=4, confusion=None, conf_dim=0):
        return lib.mv_spair_match_batch_typed(feats, dtype, B, 8, 4, 4, P16, P16, K, 3, P16, f(224.0), f(0.1), None, None,
                                              None, None, None, confusion, conf_dim, None)

    cases = [
        (lambda: typed(dtype=3), E_ARG),                                  # not an MV_FEAT_* value
        (lambda: typed(dtype=-1), E_ARG),
        (lambda: typed(dtype=3, B=0), E_ARG),                             # a bad dtype is an error even without work
        (lambda: typed(feats=None), E_ARG),
        (lambda: typed(feats=None, dtype=MV_FEAT_F16), E_ARG),
        (lambda: typed(feats=ctypes.c_void_p(17), dtype=MV_FEAT_BF16), E_ALIGN),   # odd address: not a 16-bit element
        (lambda: typed(feats=ctypes.c_void_p(17), dtype=MV_FEAT_F16), E_ALIGN),
        (lambda: typed(feats=ctypes.c_void_p(18), dtype=MV_FEAT_F32), E_ALIGN),    # 2-byte aligned is not enough for fp32
        (lambda: typed(K=65), E_RANGE),
        (lambda: typed(K=65, dtype=MV_FEAT_F16), E_RANGE),
        (lambda: typed(confusion=P16, conf_dim=3), E_ARG),                # conf_dim < K
    ]
    for call, want in cases:
        rc = call()
        assert rc == want, f"rc={rc}, wanted {want}: {lib.mv_last_error()}"
        assert b"mv_spair_match_batch_typed" in lib.mv_last_error()
    # empty work is not an error, whatever the (valid) element type; a 2-byte aligned 16-bit map is accepted
    for dtype in (MV_FEAT_F32, MV_FEAT_BF16, MV_FEAT_F16):
        assert typed(feats=None, dtype=dtype, B=0) == 0
        assert typed(feats=None, dtype=dtype, K=0) == 0
    assert typed(feats=ctypes.c_void_p(18), dtype=MV_FEAT_BF16, K=0) == 0


def test_spair_untyped_entry_point_keeps_its_messages(mv):
    """mv_spair_match_batch is the MV_FEAT_F32 case of the same launcher; its errors still name it."""
    lib = mv.load()
    P16 = ctypes.c_void_p(16)
    f = ctypes.c_float
    rc = lib.mv_spair_match_batch(P16, 2, 8, 4, 4, P16, P16, 65, 3, P16, f(224.0), f(0.1), None, None, None, None, None, None, 0,
                                  None)
    assert rc == -3
    msg = lib.mv_last_error()
    assert b"mv_spair_match_batch:" in msg and b"_typed" not in msg
