"""CPU tests of the fused dense projections' C ABI (`smt_fused_linear_forward` / `_dgrad` / `_supported`): every bad
argument is rejected with SMT_ERR_ARG and a message naming it before any device work, and T = 0 is a no-op.

The pointers are host addresses that are never dereferenced: every call below is either rejected by the argument
checks or has T = 0, so it returns before a tensor map is encoded or a kernel is launched, with or without a GPU."""
import ctypes as C

import pytest

OK, ERR_ARG = 0, -1
F32, BF16, F16 = 0, 1, 2
T_LIMIT = (1 << 31) - 512


@pytest.fixture(scope="module")
def lib(built_library):
    return built_library


_HOST_BUF = C.create_string_buffer(1 << 12)


@pytest.fixture(scope="module")
def base():
    """A 16-byte aligned host address (only its value is used)."""
    return (C.cast(_HOST_BUF, C.c_void_p).value + 15) & ~15


def _ptrs(vals):
    return (C.c_void_p * len(vals))(*vals)


def _i64(vals):
    return (C.c_int64 * len(vals))(*vals)


def _i32(vals):
    return (C.c_int * len(vals))(*vals)


def _fwd_args(base, T=300, K=512, Ns=(512, 256, 256), dtype=BF16):
    """A well-formed forward call as a dict of keyword arguments; tests break one field at a time."""
    n = len(Ns)
    return dict(x=base, ldx=K, T=T, K=K, n_seg=n, W=[base] * n, ldw=[K] * n, N=list(Ns), y=[base] * n, ldy=list(Ns),
                dtype=dtype)


def _fwd(lib, a):
    W = _ptrs(a["W"]) if a["W"] is not None else None
    ldw = _i64(a["ldw"]) if a["ldw"] is not None else None
    N = _i32(a["N"]) if a["N"] is not None else None
    y = _ptrs(a["y"]) if a["y"] is not None else None
    ldy = _i64(a["ldy"]) if a["ldy"] is not None else None
    return lib.smt_fused_linear_forward(a["x"], a["ldx"], a["T"], a["K"], a["n_seg"], W, ldw, N, y, ldy, a["dtype"],
                                        None)


def _dgrad_args(base, T=300, K=320, Ns=(320, 64, 448), dtype=BF16):
    n = len(Ns)
    return dict(dy=[base] * n, lddy=list(Ns), T=T, K=K, n_seg=n, W=[base] * n, ldw=[K] * n, N=list(Ns), dx=base, lddx=K,
                dtype=dtype)


def _dgrad(lib, a):
    dy = _ptrs(a["dy"]) if a["dy"] is not None else None
    lddy = _i64(a["lddy"]) if a["lddy"] is not None else None
    W = _ptrs(a["W"]) if a["W"] is not None else None
    ldw = _i64(a["ldw"]) if a["ldw"] is not None else None
    N = _i32(a["N"]) if a["N"] is not None else None
    return lib.smt_fused_linear_dgrad(dy, lddy, a["T"], a["K"], a["n_seg"], W, ldw, N, a["dx"], a["lddx"], a["dtype"],
                                      None)


def _rejects(lib, call, a, *words):
    assert call(lib, a) == ERR_ARG, a
    msg = lib.smt_last_error().decode()
    for w in words:
        assert w in msg, (w, msg)


def _common_rejections(lib, call, good, width_n):
    """Checks both entry points share (`check_common`)."""
    def bad(**kw):
        a = dict(good)
        a.update(kw)
        return a

    n = good["n_seg"]
    K = good["K"]
    for n_seg in (0, 4, -1):
        _rejects(lib, call, bad(n_seg=n_seg), "segments", str(n_seg))
    _rejects(lib, call, bad(dtype=F32), "16-bit")
    _rejects(lib, call, bad(dtype=3), "16-bit")
    for T in (-1, -(1 << 40), T_LIMIT, T_LIMIT + 1, 1 << 40):
        _rejects(lib, call, bad(T=T), "token count", str(T))
    for k in (0, -64, 32, K + 16, K + 1):
        _rejects(lib, call, bad(K=k), "in_features", str(k))
    _rejects(lib, call, bad(W=None), "null pointer")
    _rejects(lib, call, bad(ldw=None), "null pointer")
    _rejects(lib, call, bad(N=None), "null pointer")
    for j in range(n):
        base = good["W"][j]
        for W_j, ldw_j in ((0, K), (base + 2, K), (base + 8, K), (base, K - 64), (base, K - 1), (base, K + 1),
                           (base, K + 4), (base, 0)):
            W = list(good["W"])
            ldw = list(good["ldw"])
            W[j], ldw[j] = W_j, ldw_j
            _rejects(lib, call, bad(W=W, ldw=ldw), f"weight {j}", "16-byte aligned", "row pitch")
        for N_j in (0, -64, 32, 100, width_n[j] + 1):
            N = list(good["N"])
            N[j] = N_j
            _rejects(lib, call, bad(N=N), f"out_features {N_j} of segment {j}", "multiple of 64")


def test_forward_rejects_bad_arguments_before_any_device_work(lib, base):
    good = _fwd_args(base)
    _common_rejections(lib, _fwd, good, good["N"])

    def bad(**kw):
        a = dict(good)
        a.update(kw)
        return a

    # forward only: an N tile of 256 must not straddle two segments
    for j in range(3):
        for N_j in (64, 128, 320, 448):
            N = list(good["N"])
            N[j] = N_j
            ldy = list(good["ldy"])
            ldy[j] = max(ldy[j], N_j)
            _rejects(lib, _fwd, bad(N=N, ldy=ldy), f"out_features {N_j} of segment {j}", "multiple of 256")
    # x: null, misaligned, pitch below K or not a multiple of 16 bytes
    for x, ldx in ((0, 512), (base + 2, 512), (base + 8, 512), (base, 448), (base, 511), (base, 513), (base, 516),
                   (base, 0), (base, -512)):
        _rejects(lib, _fwd, bad(x=x, ldx=ldx), "x must be 16-byte aligned", "row pitch >= in_features")
    _rejects(lib, _fwd, bad(y=None), "null pointer")
    _rejects(lib, _fwd, bad(ldy=None), "null pointer")
    # outputs: null, misaligned, pitch below N_j or not a multiple of 16 bytes
    for j in range(3):
        for y_j, ldy_j in ((0, None), (base + 2, None), (base + 8, None), (base, -256), (base, -1), (base, 1),
                           (base, 4)):
            y = list(good["y"])
            ldy = list(good["ldy"])
            y[j] = y_j
            if ldy_j is not None:
                ldy[j] = good["N"][j] + ldy_j
            _rejects(lib, _fwd, bad(y=y, ldy=ldy), f"output {j}", "16-byte aligned", "row pitch >= out_features")
    # the last output is checked before the first map is encoded: the same rejection without a driver as with one
    y = list(good["y"])
    y[2] = base + 2
    _rejects(lib, _fwd, bad(y=y), "output 2")
    _rejects(lib, _fwd, bad(x=base + 2, y=y), "x must be")          # the first bad argument is the one reported


def test_dgrad_rejects_bad_arguments_before_any_device_work(lib, base):
    good = _dgrad_args(base)
    _common_rejections(lib, _dgrad, good, good["N"])

    def bad(**kw):
        a = dict(good)
        a.update(kw)
        return a

    # dgrad takes any N_j % 64 == 0 (the reduction may change segment at any k-block); T = 0 stops before the launch
    for j in range(3):
        N = list(good["N"])
        N[j] = 64
        assert _dgrad(lib, bad(N=N, T=0)) == OK
    _rejects(lib, _dgrad, bad(dy=None), "null pointer")
    _rejects(lib, _dgrad, bad(lddy=None), "null pointer")
    # dy_j: null, misaligned, pitch below N_j or not a multiple of 16 bytes; checked for every j before any encode
    for j in range(3):
        for dy_j, d in ((0, 0), (base + 2, 0), (base + 8, 0), (base, -64), (base, -1), (base, 1), (base, 4)):
            dy = list(good["dy"])
            lddy = list(good["lddy"])
            dy[j] = dy_j
            lddy[j] = good["N"][j] + d
            _rejects(lib, _dgrad, bad(dy=dy, lddy=lddy), f"dy {j}", "16-byte aligned", "row pitch >= out_features")
    # dx: null, misaligned, pitch below K or not a multiple of 16 bytes
    for dx, d in ((0, 0), (base + 2, 0), (base + 8, 0), (base, -64), (base, -1), (base, 1), (base, 4)):
        _rejects(lib, _dgrad, bad(dx=dx, lddx=good["K"] + d), "dx must be 16-byte aligned", "row pitch >= in_features")


@pytest.mark.parametrize("dtype", [BF16, F16])
def test_zero_tokens_is_a_no_op(lib, base, dtype):
    """T = 0 returns SMT_OK before any tensor map or launch, even with null activation and output pointers (what
    `ops` passes for an empty batch); the weights and sizes are still checked."""
    a = _fwd_args(base, T=0, dtype=dtype)
    assert _fwd(lib, a) == OK
    a.update(x=None, y=[0, 0, 0], ldy=[0, 0, 0], ldx=0)
    assert _fwd(lib, a) == OK
    a.update(y=None, ldy=None)
    assert _fwd(lib, a) == OK
    _rejects(lib, _fwd, dict(a, K=96), "in_features")
    d = _dgrad_args(base, T=0, dtype=dtype)
    assert _dgrad(lib, d) == OK
    d.update(dy=None, lddy=None, dx=None, lddx=0)
    assert _dgrad(lib, d) == OK
    _rejects(lib, _dgrad, dict(d, n_seg=4), "segments")


def test_supported_truth_table(lib):
    sup = lib.smt_fused_linear_supported

    def s(Ns, K=4096, dtype=BF16, dgrad=0, n_seg=None):
        N = _i32(Ns) if Ns is not None else None
        return sup(len(Ns) if n_seg is None else n_seg, N, K, dtype, dgrad)

    for dgrad in (0, 1):
        # accepted: 1..3 segments of 16-bit weights, K % 64 == 0, N_j % 256 == 0
        for Ns in ([4096], [4096, 1024, 1024], [256, 256], [128256], [8192, 1024, 1024]):
            for dtype in (BF16, F16):
                assert s(Ns, dtype=dtype, dgrad=dgrad) == 1, (Ns, dtype, dgrad)
        assert s([256], K=64, dgrad=dgrad) == 1
        assert s([256], K=14336, dgrad=dgrad) == 1
        # rejected in both directions
        assert s([256], dtype=F32, dgrad=dgrad) == 0
        assert s([256], dtype=3, dgrad=dgrad) == 0
        assert s([256], dtype=-1, dgrad=dgrad) == 0
        for K in (0, -64, 32, 4100, 4097):
            assert s([256], K=K, dgrad=dgrad) == 0, K
        assert s([], dgrad=dgrad) == 0
        assert s([256] * 4, dgrad=dgrad) == 0
        assert s([256], n_seg=-1, dgrad=dgrad) == 0
        assert sup(1, None, 4096, BF16, dgrad) == 0
        for bad in (0, -256, 32, 100, 257):
            assert s([256, bad], dgrad=dgrad) == 0, bad
            assert s([bad, 256, 256], dgrad=dgrad) == 0, bad
    # N_j % 64 == 0 but not % 256: input gradient only (a forward N tile would straddle two segments)
    for Ns in ([64], [128], [192], [320, 64, 448], [4096, 64]):
        assert s(Ns, dgrad=1) == 1, Ns
        assert s(Ns, dgrad=0) == 0, Ns
