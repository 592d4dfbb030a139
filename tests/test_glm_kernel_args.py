"""Argument checks of the batched GLM entry points without a GPU: X'R rejects a misaligned R or workspace, and an
empty row slice (T = 0) accepts null row pointers but still rejects null outputs and workspaces.  Every call below
fails its argument checks before any CUDA call."""
import ctypes

import _sglm_native as nat

E_INVALID, E_SHAPE, E_ALIGN, E_WORKSPACE = -1, -2, -3, -4


def test_pb_xt_r_rejects_misaligned_r_and_workspace():
    lib = nat.lib()
    p = ctypes.c_void_p(64)              # 16-byte aligned, never dereferenced
    odd = ctypes.c_void_p(64 + 8)        # 8 bytes off: R and the workspace are read / written as double2
    big = 1 << 40
    assert lib.sglm_pb_xt_r_f64(p, 8, 100, 8, odd, 64, p, p, big, None) == E_ALIGN
    assert b"alignment" in lib.sglm_last_error()
    assert lib.sglm_pb_xt_r_f64(p, 8, 100, 8, p, 64, p, odd, big, None) == E_ALIGN
    # X may be misaligned (the GEMM loads it by scalars then); the shape, pointer and size checks still apply
    assert lib.sglm_pb_xt_r_f64(odd, 8, 100, 8, p, 64, p, p, 8, None) == E_WORKSPACE
    assert lib.sglm_pb_xt_r_f64(p, 8, 100, 8, p, 96, p, p, big, None) == E_SHAPE
    assert lib.sglm_pb_xt_r_f64(p, 8, 100, 8, None, 64, p, p, big, None) == E_INVALID
    assert lib.sglm_pb_xt_r_f64(None, 8, 100, 8, p, 64, p, p, big, None) == E_INVALID


def test_empty_row_slice_still_needs_outputs_and_workspace():
    lib = nat.lib()
    p = ctypes.c_void_p(64)
    big = 1 << 40
    # sglm_pb_xt_r_f64: T = 0 with X = R = NULL gets past the pointer check only with Gw and the workspace
    assert lib.sglm_pb_xt_r_f64(None, 8, 0, 8, None, 64, None, p, big, None) == E_INVALID
    assert lib.sglm_pb_xt_r_f64(None, 8, 0, 8, None, 64, p, None, big, None) == E_INVALID
    assert lib.sglm_pb_xt_r_f64(None, 8, 0, 8, None, 64, p, ctypes.c_void_p(72), big, None) == E_ALIGN
    assert lib.sglm_pb_xt_r_f64(None, 8, 0, 8, None, 64, p, p, 8, None) == E_WORKSPACE
    # sglm_xt_vec_f64
    assert lib.sglm_xt_vec_f64(None, 8, None, 0, 8, None, p, big, None) == E_INVALID
    assert lib.sglm_xt_vec_f64(None, 8, None, 0, 8, p, None, big, None) == E_INVALID
    assert lib.sglm_xt_vec_f64(None, 8, p, 5, 8, p, p, big, None) == E_INVALID         # T > 0: X is needed
    assert lib.sglm_xt_vec_f64(p, 8, None, 5, 8, p, p, big, None) == E_INVALID
    # sglm_score_glm_f64 (X, y, rw, T, C, w, b, power, resid, sums, workspace)
    for power in (1.0, 2.0, 1.5):
        assert lib.sglm_score_glm_f64(None, 8, None, None, 0, 8, p, p, power, None, None, p, None) == E_INVALID
        assert lib.sglm_score_glm_f64(None, 8, None, None, 0, 8, p, p, power, None, p, None, None) == E_INVALID
        assert lib.sglm_score_glm_f64(None, 8, None, None, 0, 8, None, p, power, None, p, p, None) == E_INVALID
        assert lib.sglm_score_glm_f64(None, 8, p, None, 3, 8, p, p, power, None, p, p, None) == E_INVALID
        assert lib.sglm_score_glm_f64(p, 8, None, None, 3, 8, p, p, power, None, p, p, None) == E_INVALID
    # sglm_glm_irls_prepare_f64 (X, y, rw, T, C, w, b, power, weight, z, sums, workspace)
    for power in (1.0, 2.0, 3.0):
        assert lib.sglm_glm_irls_prepare_f64(None, 8, None, None, 0, 8, p, p, power, None, None, None, p,
                                             None) == E_INVALID
        assert lib.sglm_glm_irls_prepare_f64(None, 8, None, None, 0, 8, p, p, power, None, None, p, None,
                                             None) == E_INVALID
        assert lib.sglm_glm_irls_prepare_f64(p, 8, p, None, 3, 8, p, p, power, None, p, p, p, None) == E_INVALID
        assert lib.sglm_glm_irls_prepare_f64(p, 8, p, None, 3, 8, p, p, power, p, None, p, p, None) == E_INVALID
    # sglm_glm_epilogue_f64 (Eta, ldb, n, T, Y, ldy, ycol, RW, ldrw, rw_a, rw_b, b, status, power, mode, sums, ws)
    for mode in (0, 1):
        rw_b = p if mode else None
        args = lambda eta=None, y=None, ycol=p, rw_a=p, b=p, sums=p, ws=p, T=0, rw_b=rw_b: (
            eta, 64, 5, T, y, 1, ycol, None, 0, rw_a, rw_b, b, None, 1.5, mode, sums, ws, big, None)
        assert lib.sglm_glm_epilogue_f64(*args(sums=None)) == E_INVALID
        assert lib.sglm_glm_epilogue_f64(*args(ws=None)) == E_INVALID
        assert lib.sglm_glm_epilogue_f64(*args(ycol=None)) == E_INVALID
        assert lib.sglm_glm_epilogue_f64(*args(rw_a=None)) == E_INVALID
        assert lib.sglm_glm_epilogue_f64(*args(b=None)) == E_INVALID
        assert lib.sglm_glm_epilogue_f64(*args(T=4, y=p)) == E_INVALID                  # T > 0: Eta is needed
        assert lib.sglm_glm_epilogue_f64(*args(T=4, eta=p)) == E_INVALID                # ... and Y
        if mode:
            assert lib.sglm_glm_epilogue_f64(*args(rw_b=None)) == E_INVALID
        assert lib.sglm_pb_epilogue_f64(None, 64, 5, 0, None, 1, p, None, 0, p, rw_b, p, None, mode, None, p, big,
                                        None) == E_INVALID
