"""Argument checks of the row-sharded GLM entry points without a GPU: the staged weighted tcgen05 Gram and the
fixed-order sum of gathered partials reject bad shapes, missing pointers and unsupported plans before any CUDA call."""
import ctypes

import _sglm_native as nat


def test_row_sharded_glm_entry_points_validate_before_cuda():
    lib = nat.lib()
    p = ctypes.c_void_p(64)        # never dereferenced: every call below fails its argument checks first
    colS = (ctypes.c_int32 * 11)(*([1] * 11))
    sizes = (ctypes.c_int64 * 1)(100)
    member = (ctypes.c_int32 * 1)(1)
    # sglm_gram_tc_colstats_scaled_f64: shape, null outputs, a missing row scale (allowed only for an empty slice)
    assert lib.sglm_gram_tc_colstats_scaled_f64(p, 8, p, 1, 1, -1, 8, p, p, p, None) == -2
    assert b"bad shape" in lib.sglm_last_error()
    assert lib.sglm_gram_tc_colstats_scaled_f64(p, 4, p, 1, 1, 100, 8, p, p, p, None) == -2
    assert lib.sglm_gram_tc_colstats_scaled_f64(p, 8, p, 1, 1, 100, 8, p, None, p, None) == -1
    assert lib.sglm_gram_tc_colstats_scaled_f64(p, 8, p, 1, 1, 100, 8, None, p, p, None) == -1
    assert b"null" in lib.sglm_last_error()
    # sglm_gram_tc_scaled_partial_f64: membership, cell count, row scale, then the shared shape / pointer checks
    args = lambda T=100, ldx=8, rs=p, n_cells=1, n_out=1, mem=member, ws=p: (
        p, ldx, p, 1, 1, T, 8, rs, p, p, colS, n_cells, sizes, p, n_out, mem, ws, 1 << 30, None)
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(n_out=0)) == -1
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(mem=None)) == -1
    assert b"membership" in lib.sglm_last_error()
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(n_cells=257)) == -6
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(rs=None)) == -1
    assert b"row_scale" in lib.sglm_last_error()
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(T=-1)) == -2
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(ldx=4)) == -2
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(ws=None)) == -1
    assert lib.sglm_gram_tc_scaled_partial_f64(*args(ws=ctypes.c_void_p(64 + 8))) == -3      # 1024-byte alignment
    # sglm_reduce_parts_f64
    assert lib.sglm_reduce_parts_f64(p, 10, 0, p, None) == -2
    assert lib.sglm_reduce_parts_f64(p, -1, 2, p, None) == -2
    assert lib.sglm_reduce_parts_f64(None, 10, 2, p, None) == -1
    assert lib.sglm_reduce_parts_f64(p, 10, 2, None, None) == -1
    assert lib.sglm_reduce_parts_f64(None, 0, 2, None, None) == 0         # nothing to add: no launch
