"""CPU tests of the decoder-layer entry points `smt_rmsnorm_*`, `smt_rope_*` and `smt_swiglu_*`: every argument
they reject is rejected before any memory is touched, so these run on host pointers without a device.  Also the
norm width limit that `decoder_fusion` shares with the C code."""
import ctypes

import pytest


def _p(buf):
    return ctypes.cast(buf, ctypes.c_void_p).value


@pytest.fixture(scope="module")
def lib(built_library):
    return built_library


@pytest.fixture(scope="module")
def b():
    """A 16-byte aligned host address with room for every tensor the rejected calls below could name."""
    buf = ctypes.create_string_buffer(8192 + 16)
    yield (_p(buf) + 15) & ~15


def _rejected(ret, lib, what):
    assert ret == -1
    assert what in lib.smt_last_error(), lib.smt_last_error()


# ---- RMSNorm -------------------------------------------------------------------------------------------------------

def _norm_fwd(lib, a, res, w, T, H, h_out, y, rstd):
    return lib.smt_rmsnorm_forward(a, res, w, T, H, 1e-6, h_out, y, rstd, None)


def _norm_bwd(lib, x, w, rstd, dy, dres, T, H, dx):
    return lib.smt_rmsnorm_backward(x, w, rstd, dy, dres, T, H, dx, None)


def test_rmsnorm_rejects_bad_arguments_without_a_device(lib, b):
    # a negative row count, and widths that are not a positive multiple of 8 or exceed 32 768
    for T, H in ((-1, 64), (1, 0), (1, -8), (1, 12), (1, 4), (1, 32776), (1, 65536), (0, 12), (0, 32776)):
        _rejected(_norm_fwd(lib, b, b, b, T, H, b, b, b), lib, b"multiple of 8")
        _rejected(_norm_bwd(lib, b, b, b, b, b, T, H, b), lib, b"multiple of 8")
    # every pointer the forward needs, null in turn (h_out only with a residual)
    for i in range(4):
        args = [b] * 4
        args[i] = None
        a, w, y, rstd = args
        _rejected(_norm_fwd(lib, a, None, w, 1, 64, None, y, rstd), lib, b"null pointer")
        _rejected(_norm_fwd(lib, a, b, w, 1, 64, b, y, rstd), lib, b"null pointer")
    _rejected(_norm_fwd(lib, b, b, b, 1, 64, None, b, b), lib, b"null pointer")
    # every pointer of the backward but dres, null in turn
    for i in range(5):
        args = [b] * 5
        args[i] = None
        x, w, rstd, dy, dx = args
        _rejected(_norm_bwd(lib, x, w, rstd, dy, None, 1, 64, dx), lib, b"null pointer")
        _rejected(_norm_bwd(lib, x, w, rstd, dy, b, 1, 64, dx), lib, b"null pointer")
    # a tensor off the 16-byte grid, rstd off the 4-byte grid
    for i in range(6):
        args = [b] * 6
        args[i] = b + 2
        a, res, w, h_out, y, rstd = args
        _rejected(_norm_fwd(lib, a, res, w, 1, 64, h_out, y, rstd), lib, b"aligned")
    for i in range(6):
        args = [b] * 6
        args[i] = b + 2
        x, w, rstd, dy, dres, dx = args
        _rejected(_norm_bwd(lib, x, w, rstd, dy, dres, 1, 64, dx), lib, b"aligned")
    # no rows is a no-op, even with null pointers
    assert _norm_fwd(lib, None, None, None, 0, 64, None, None, None) == 0
    assert _norm_fwd(lib, None, b, None, 0, 32768, None, None, None) == 0
    assert _norm_bwd(lib, None, None, None, None, None, 0, 8, None) == 0


def test_norm_width_limit_agrees_with_the_c_limit(lib):
    """`decoder_fusion` sends a norm to the kernels only up to `_MAX_NORM_WIDTH`; the C entry points take exactly
    that width and refuse the next multiple of 8."""
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    n = D._MAX_NORM_WIDTH
    assert n == 32768
    assert _norm_fwd(lib, None, None, None, 0, n, None, None, None) == 0
    assert _norm_bwd(lib, None, None, None, None, None, 0, n, None) == 0
    _rejected(_norm_fwd(lib, None, None, None, 0, n + 8, None, None, None), lib, b"32768")
    _rejected(_norm_bwd(lib, None, None, None, None, None, 0, n + 8, None), lib, b"32768")


# ---- RoPE ----------------------------------------------------------------------------------------------------------

def _rope(lib, bwd, q, k, cos, sin, B, S, Hq, Hk, bstride, qo, ko):
    fn = lib.smt_rope_backward if bwd else lib.smt_rope_forward
    return fn(q, k, cos, sin, B, S, Hq, Hk, bstride, qo, ko, None)


@pytest.mark.parametrize("bwd", [False, True])
def test_rope_rejects_bad_arguments_without_a_device(lib, b, bwd):
    # negative shapes and a cos/sin batch stride that is negative or not a multiple of 8
    for shape in ((-1, 1, 1, 1, 0), (1, -1, 1, 1, 0), (1, 1, -1, 1, 0), (1, 1, 1, -1, 0), (1, 1, 1, 1, -8),
                  (2, 1, 1, 1, 12), (0, 1, 1, 1, 4)):
        _rejected(_rope(lib, bwd, b, b, b, b, *shape, b, b), lib, b"bad shape")
    # every pointer null in turn
    for i in range(6):
        args = [b] * 6
        args[i] = None
        q, k, cos, sin, qo, ko = args
        _rejected(_rope(lib, bwd, q, k, cos, sin, 1, 1, 1, 1, 0, qo, ko), lib, b"null pointer")
    # a tensor off the 16-byte grid
    for i in range(6):
        args = [b] * 6
        args[i] = b + 8
        q, k, cos, sin, qo, ko = args
        _rejected(_rope(lib, bwd, q, k, cos, sin, 1, 1, 1, 1, 0, qo, ko), lib, b"aligned")
    # no rows is a no-op, even with null pointers
    for shape in ((0, 4, 2, 1, 0), (2, 0, 2, 1, 0), (2, 4, 0, 0, 0)):
        assert _rope(lib, bwd, None, None, None, None, *shape, None, None) == 0


# ---- SwiGLU --------------------------------------------------------------------------------------------------------

def test_swiglu_rejects_bad_arguments_without_a_device(lib, b):
    for n in (-8, -1, 1, 4, 12, 1001):
        _rejected(lib.smt_swiglu_forward(b, b, n, b, None), lib, b"multiple of 8")
        _rejected(lib.smt_swiglu_backward(b, b, b, n, b, b, None), lib, b"multiple of 8")
    for i in range(3):
        args = [b] * 3
        args[i] = None
        g, u, h = args
        _rejected(lib.smt_swiglu_forward(g, u, 8, h, None), lib, b"null pointer")
        args[i] = b + 4
        g, u, h = args
        _rejected(lib.smt_swiglu_forward(g, u, 8, h, None), lib, b"aligned")
    for i in range(5):
        args = [b] * 5
        args[i] = None
        g, u, dh, dg, du = args
        _rejected(lib.smt_swiglu_backward(g, u, dh, 8, dg, du, None), lib, b"null pointer")
        args[i] = b + 4
        g, u, dh, dg, du = args
        _rejected(lib.smt_swiglu_backward(g, u, dh, 8, dg, du, None), lib, b"aligned")
    assert lib.smt_swiglu_forward(None, None, 0, None, None) == 0
    assert lib.smt_swiglu_backward(None, None, None, 0, None, None, None) == 0
