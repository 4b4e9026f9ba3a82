"""GPU tests of the fused dense GEMMs (`csrc/dense_gemm.cu`): the q/k/v forward `y_j = x W_j^T`, the q/k/v input gradient
`dx = sum_j dy_j W_j`, and the lm-head GEMMs of the fused loss (N = 128 256).

Every element is checked against an fp64 product of the same 16-bit inputs, with a bound made of one rounding to the
output type at that element plus a wide fp32-accumulation term, so a wrong small-magnitude element cannot hide behind
the tensor's largest one. The rounding must be unbiased (round to nearest, not toward zero). The shapes reach the
kernel's edges: one k-block, a wrapping 6-stage ring, a segment change at every stage, a raster group after a full group
of 16 M tiles, one tile more than the resident CTA pairs, and the lm-head's odd N-tile counts. Segmentation and row
splits must not change a single bit; strided operands with NaN padding and sentinel-filled output guard bands show that
the kernel reads and writes only inside the logical bounds; a NaN or Inf input spoils only the outputs it feeds."""
import ctypes as C
import math
import zlib

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16, F16 = torch.bfloat16, torch.float16
_FRAC_BITS = {BF16: 7, F16: 10}
_MIN_NORMAL_EXP = {BF16: -126, F16: -14}
ACC_COEF = 2.0 ** -20              # fp32 accumulation term: ACC_COEF * sqrt(K_red) * (|a| @ |b|)
BIAS_MIN_ELEMS = 10 ** 6           # outputs at least this large also get the rounding-bias check
BIAS_LIMIT = 0.02                  # round to nearest: ~0 (spread ~3e-4 at 1e6 elements); toward zero: ~-0.5
SENTINEL = -12345                  # int16 bit pattern of the output guard bands
CHUNK = 16384                      # rows of W per fp64 reference product


@pytest.fixture(scope="module")
def ops(built_library):
    from sparse_matrix_tuning_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def lib(built_library):
    return built_library


def _case(T, K, Ns, dtype):
    return pytest.param(T, K, Ns, dtype, id=f"{T}x{K}-{'+'.join(map(str, Ns))}-{str(dtype)[6:]}")


# (T, K, N_j, dtype); forward: K = reduction, N_j = output widths (multiples of 256)
FWD_CASES = [
    _case(1, 64, [256], BF16),                              # one token, one k-block, one tile; rank 1 fully out of bounds
    _case(129, 448, [256, 256, 256], F16),                  # 7 k-blocks: the 6-stage ring wraps; three one-tile segments
    _case(255, 384, [512, 256], BF16),                      # exactly 6 k-blocks
    _case(4097, 1024, [1024, 256, 256], BF16),              # 17 M tiles: a full raster group of 16, then a group of 1
    _case(8449, 4096, [4096, 1024, 1024], BF16),            # LLaMA-3-8B q/k/v, 34 M tiles
    _case(18945, 256, [256], BF16),                         # 75 tiles: one more than 74 CTA pairs
    _case(2048, 4096, [4096, 4096, 4096], BF16),            # LLaMA-2-7B q/k/v (MHA)
    _case(1000, 8192, [8192, 1024, 1024], BF16),            # LLaMA-3-70B q/k/v
    _case(513, 14336, [4096], F16),                         # 224 k-blocks
    _case(2048, 4096, [128256], BF16),                      # LLaMA-3 lm-head: 501 N tiles
    _case(600, 4096, [32000], BF16),                        # LLaMA-2 lm-head: 125 N tiles
]

# (T, K = width of dx, N_j = reduction segments, dtype)
DGRAD_CASES = [
    _case(1, 64, [64], BF16),                               # one k-block, one 64-column chunk
    _case(129, 192, [64, 64, 64], F16),                     # the segment changes at every stage
    _case(300, 320, [320, 64, 448], BF16),                  # 13 k-blocks, segment ends inside and at the end of the ring;
                                                            # dx = one tile + 64 columns
    _case(4097, 1024, [1024, 256, 256], BF16),              # the raster edge
    _case(18945, 64, [256], BF16),                          # 75 tiles
    _case(1000, 8192, [8192, 1024, 1024], BF16),            # LLaMA-3-70B
    _case(2048, 4096, [128256], BF16),                      # lm-head input gradient: 2 004 k-blocks
]


# ---- inputs and the fp64 reference -------------------------------------------------------------------------------------

def _gen(*key):
    g = torch.Generator(device="cuda")
    g.manual_seed(zlib.crc32(repr(key).encode()))
    return g


def _operand(rows, cols, dtype, g, scale=1.0, spread_rows=False, spread_cols=False):
    """randn * scale, with rows and/or columns multiplied by powers of two in 2^-4 .. 2^3, so that the outputs span many
    binades and an element-wise bound is tested at small magnitudes too."""
    t = torch.randn(rows, cols, device="cuda", generator=g) * scale
    if spread_rows:
        t *= torch.exp2(torch.randint(-4, 4, (rows, 1), device="cuda", generator=g).float())
    if spread_cols:
        t *= torch.exp2(torch.randint(-4, 4, (1, cols), device="cuda", generator=g).float())
    return t.to(dtype)


def _fwd_inputs(T, K, Ns, dtype):
    g = _gen("fwd", T, K, tuple(Ns), str(dtype))
    x = _operand(T, K, dtype, g, spread_rows=True)
    ws = [_operand(n, K, dtype, g, scale=K ** -0.5, spread_rows=True) for n in Ns]
    return x, ws


def _dgrad_inputs(T, K, Ns, dtype):
    g = _gen("dgrad", T, K, tuple(Ns), str(dtype))
    dys = [_operand(T, n, dtype, g, spread_rows=True) for n in Ns]
    ws = [_operand(n, K, dtype, g, scale=sum(Ns) ** -0.5, spread_cols=True) for n in Ns]
    return dys, ws


def _fwd_reference(x, w):
    """Column chunks (s, x @ w[s:e]^T, |x| @ |w[s:e]|^T) in fp64."""
    xd = x.double()
    xa = xd.abs()
    for s in range(0, w.shape[0], CHUNK):
        wd = w[s:s + CHUNK].double()
        yield s, xd @ wd.t(), xa @ wd.abs().t()


def _dgrad_reference(dys, ws):
    """(sum_j dy_j @ w_j, sum_j |dy_j| @ |w_j|) in fp64."""
    ref = absref = 0
    for dy, w in zip(dys, ws):
        for s in range(0, w.shape[0], CHUNK):
            a, b = dy[:, s:s + CHUNK].double(), w[s:s + CHUNK].double()
            ref = ref + a @ b
            absref = absref + a.abs() @ b.abs()
    return ref, absref


def _ulp(a, dtype):
    """Spacing of `dtype` numbers at |a| (fp64), the subnormal spacing below the smallest normal."""
    p, emin = _FRAC_BITS[dtype], _MIN_NORMAL_EXP[dtype]
    _, e = torch.frexp(a)                                   # a = m 2^e, m in [0.5, 1)
    e = torch.where(a >= 2.0 ** emin, e - 1, emin) - p      # exponent of the spacing
    return ((e.long() + 1023) << 52).view(torch.float64)    # 2^e, built from its bits


class _Bound:
    """|got - ref| <= ulp_out(|ref|) + ACC_COEF * sqrt(K_red) * (|a| @ |b|) for every element of one output, checked chunk
    by chunk; also collects the largest error / bound ratio and the rounding bias mean((|got| - |ref|) / ulp_out)."""

    def __init__(self, name, dtype, k_red):
        self.name, self.dtype, self.acc = name, dtype, ACC_COEF * math.sqrt(k_red)
        self.ratio, self.bias_sum, self.n = 0.0, 0.0, 0

    def check(self, got, ref, absref, col0=0):
        assert got.shape == ref.shape
        g = got.double()
        ulp = _ulp(ref.abs(), self.dtype)
        err = (g - ref).abs()
        bound = ulp + self.acc * absref
        bad = ~(err <= bound)                               # NaN fails too
        if bad.any():
            r, c = [int(i) for i in bad.nonzero()[0]]
            raise AssertionError(f"{self.name}: {int(bad.sum())} elements outside the bound; first at "
                                 f"[{r}, {col0 + c}]: got {g[r, c].item()!r}, fp64 {ref[r, c].item()!r}, "
                                 f"bound {bound[r, c].item()!r}")
        self.ratio = max(self.ratio, (err / bound).max().item())
        self.bias_sum += ((g.abs() - ref.abs()) / ulp).sum().item()
        self.n += got.numel()

    def finish(self):
        """Prints the headroom (shown with `pytest -s`) and checks the rounding bias of outputs large enough for it."""
        line = f"{self.name}: max error / bound {self.ratio:.4f}"
        if self.n >= BIAS_MIN_ELEMS:
            bias = self.bias_sum / self.n
            print(f"{line}, rounding bias {bias:+.5f} ulp over {self.n} elements")
            assert abs(bias) <= BIAS_LIMIT, f"{self.name}: rounding bias {bias:.4f} ulp over {self.n} elements"
        else:
            print(line)


# ---- element-wise sweeps against fp64 ----------------------------------------------------------------------------------

@pytest.mark.parametrize("T,K,Ns,dtype", FWD_CASES)
def test_forward_vs_fp64(ops, T, K, Ns, dtype):
    x, ws = _fwd_inputs(T, K, Ns, dtype)
    assert ops.fused_linear_supported(ws)
    ys = ops.fused_linear_forward(x, ws)
    again = ops.fused_linear_forward(x, ws)
    for j, (y, y2, w) in enumerate(zip(ys, again, ws)):
        assert y.shape == (T, w.shape[0]) and y.dtype == dtype
        assert torch.equal(y, y2), f"y_{j} differs between two identical calls"
        b = _Bound(f"y{j}", dtype, K)
        for s, ref, absref in _fwd_reference(x, w):
            b.check(y[:, s:s + ref.shape[1]], ref, absref, s)
        b.finish()


@pytest.mark.parametrize("T,K,Ns,dtype", DGRAD_CASES)
def test_dgrad_vs_fp64(ops, T, K, Ns, dtype):
    dys, ws = _dgrad_inputs(T, K, Ns, dtype)
    assert ops.fused_linear_supported(ws, dgrad=True)
    dx = ops.fused_linear_dgrad(dys, ws)
    assert dx.shape == (T, K) and dx.dtype == dtype
    assert torch.equal(dx, ops.fused_linear_dgrad(dys, ws)), "dx differs between two identical calls"
    ref, absref = _dgrad_reference(dys, ws)
    b = _Bound("dx", dtype, sum(Ns))
    b.check(dx, ref, absref)
    b.finish()


# ---- exact invariances ------------------------------------------------------------------------------------------------

def _bits(t):
    return t.view(torch.int16)


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


@pytest.mark.parametrize("T,K,Ns,dtype", [FWD_CASES[1], FWD_CASES[3], FWD_CASES[4]])
def test_forward_segmentation_is_exact(ops, T, K, Ns, dtype):
    """Three segments compute what one segment of the concatenated weight does, column for column: the k order is the
    same, only the segment bookkeeping (first tile, output pointer and pitch) differs."""
    x, ws = _fwd_inputs(T, K, Ns, dtype)
    whole = ops.fused_linear_forward(x, [torch.cat(ws)])[0]
    for j, (y, part) in enumerate(zip(ops.fused_linear_forward(x, ws), whole.split(Ns, dim=1))):
        assert _same_bits(y, part), f"segment {j}"


@pytest.mark.parametrize("T,K,Ns,dtype", [DGRAD_CASES[1], DGRAD_CASES[2], DGRAD_CASES[3]])
def test_dgrad_segmentation_is_exact(ops, T, K, Ns, dtype):
    """The reduction through three (dy_j, W_j) segments equals one segment of the concatenations: same k-blocks in the
    same order into one fp32 accumulator."""
    dys, ws = _dgrad_inputs(T, K, Ns, dtype)
    got = ops.fused_linear_dgrad(dys, ws)
    assert _same_bits(got, ops.fused_linear_dgrad([torch.cat(dys, dim=1)], [torch.cat(ws)]))


# offsets 256 and 2048 keep every row in its CTA and TMEM lane (the loss's 2048-row chunks rely on them); 1 and 129 move
# rows to the other CTA of the pair and to other TMEM lanes
SPLITS = [(0, 1), (1, 129), (129, 256), (1, 4097), (129, 4097), (256, 4097), (256, 2048), (2048, 4097), (0, 2048)]


def test_forward_row_splits_are_exact(ops):
    T, K, Ns, dtype = 4097, 1024, [1024, 256, 256], BF16
    x, ws = _fwd_inputs(T, K, Ns, dtype)
    whole = ops.fused_linear_forward(x, ws)
    for s, e in SPLITS:
        for j, (y, part) in enumerate(zip(whole, ops.fused_linear_forward(x[s:e], ws))):
            assert _same_bits(y[s:e], part), (s, e, j)


def test_dgrad_row_splits_are_exact(ops):
    """Also through `out=`, a row slice of a larger buffer, as the fused loss writes dh."""
    T, K, Ns, dtype = 4097, 1024, [1024, 256, 256], BF16
    dys, ws = _dgrad_inputs(T, K, Ns, dtype)
    whole = ops.fused_linear_dgrad(dys, ws)
    for s, e in SPLITS:
        part = ops.fused_linear_dgrad([dy[s:e] for dy in dys], ws)
        assert _same_bits(whole[s:e], part), (s, e)
    into = torch.full_like(whole, float("nan"))
    for s, e in ((0, 1), (1, 129), (129, 2048), (2048, 4097)):
        ops.fused_linear_dgrad([dy[s:e] for dy in dys], ws, out=into[s:e])
    assert _same_bits(into, whole)


# ---- strided operands and guard bands (C ABI: `ops` allocates contiguous outputs) ----------------------------------------

def _padded_input(t):
    """`t` copied into a NaN-filled buffer with 256 more rows and a row pitch of width + 64; returns the view."""
    rows, cols = t.shape
    buf = torch.full((rows + 256, cols + 64), float("nan"), dtype=t.dtype, device=t.device)
    buf[:rows, :cols] = t
    return buf[:rows, :cols]


def _guarded_output(rows, cols, dtype):
    """(buffer, view): the [rows, cols] view has a row pitch of cols + 64 and 256 rows after it, all SENTINEL."""
    buf = torch.full((rows + 256, cols + 64), SENTINEL, dtype=torch.int16, device="cuda").view(dtype)
    return buf, buf[:rows, :cols]


def _assert_guard_intact(buf, rows, cols, what):
    outside = _bits(buf).clone()
    outside[:rows, :cols] = SENTINEL
    n = int((outside != SENTINEL).sum())
    assert n == 0, f"{what}: {n} elements written outside the [{rows}, {cols}] output"


def _seg(vals, ctype):
    return (ctype * len(vals))(*vals)


@pytest.mark.parametrize("T,K,Ns,dtype", [FWD_CASES[0], FWD_CASES[1], FWD_CASES[3]])
def test_forward_strided_operands_and_guard_bands(ops, lib, T, K, Ns, dtype):
    from sparse_matrix_tuning_b200._lib import dtype_id, stream_ptr
    x, ws = _fwd_inputs(T, K, Ns, dtype)
    want = ops.fused_linear_forward(x, ws)
    xp, wps = _padded_input(x), [_padded_input(w) for w in ws]
    outs = [_guarded_output(T, n, dtype) for n in Ns]
    rc = lib.smt_fused_linear_forward(
        xp.data_ptr(), xp.stride(0), T, K, len(Ns), _seg([w.data_ptr() for w in wps], C.c_void_p),
        _seg([w.stride(0) for w in wps], C.c_int64), _seg(Ns, C.c_int), _seg([v.data_ptr() for _, v in outs], C.c_void_p),
        _seg([v.stride(0) for _, v in outs], C.c_int64), dtype_id(dtype), stream_ptr())
    assert rc == 0, lib.smt_last_error()
    for j, ((buf, view), y) in enumerate(zip(outs, want)):
        assert view.stride(0) == Ns[j] + 64 and xp.stride(0) == K + 64
        assert _same_bits(view, y), f"y_{j} with strided operands differs from the contiguous call"
        _assert_guard_intact(buf, T, Ns[j], f"y_{j}")


@pytest.mark.parametrize("T,K,Ns,dtype", [DGRAD_CASES[0], DGRAD_CASES[1], DGRAD_CASES[2], DGRAD_CASES[3]])
def test_dgrad_strided_operands_and_guard_bands(ops, lib, T, K, Ns, dtype):
    from sparse_matrix_tuning_b200._lib import dtype_id, stream_ptr
    dys, ws = _dgrad_inputs(T, K, Ns, dtype)
    want = ops.fused_linear_dgrad(dys, ws)
    dyps, wps = [_padded_input(dy) for dy in dys], [_padded_input(w) for w in ws]
    buf, dx = _guarded_output(T, K, dtype)
    rc = lib.smt_fused_linear_dgrad(
        _seg([d.data_ptr() for d in dyps], C.c_void_p), _seg([d.stride(0) for d in dyps], C.c_int64), T, K, len(Ns),
        _seg([w.data_ptr() for w in wps], C.c_void_p), _seg([w.stride(0) for w in wps], C.c_int64), _seg(Ns, C.c_int),
        dx.data_ptr(), dx.stride(0), dtype_id(dtype), stream_ptr())
    assert rc == 0, lib.smt_last_error()
    assert _same_bits(dx, want), "dx with strided operands differs from the contiguous call"
    _assert_guard_intact(buf, T, K, "dx")


# ---- non-finite inputs ------------------------------------------------------------------------------------------------

def _assert_local(got, clean, ref, what):
    """Non-finite exactly where the fp64 reference is, and every other element bit-identical to the clean run."""
    fin = torch.isfinite(ref)
    assert torch.equal(torch.isfinite(got), fin), f"{what}: non-finite pattern differs from fp64"
    assert not fin.all(), f"{what}: the poisoned inputs should reach this output"
    assert torch.equal(_bits(got)[fin], _bits(clean)[fin]), f"{what}: a finite element changed"


@pytest.mark.parametrize("T,K,Ns,dtype", [FWD_CASES[1], FWD_CASES[3]])
def test_forward_non_finite_inputs_stay_local(ops, T, K, Ns, dtype):
    x, ws = _fwd_inputs(T, K, Ns, dtype)
    clean = ops.fused_linear_forward(x, ws)
    x = x.clone()
    ws = [w.clone() for w in ws]
    x[0, 0] = float("nan")                                  # first row, first k-block
    x[T - 1, K - 1] = float("inf")                          # last row (last M tile), last k-block
    ws[1][Ns[1] - 1, K // 2] = float("nan")                 # segment 1, last column
    got = ops.fused_linear_forward(x, ws)
    for j, (y, c, w) in enumerate(zip(got, clean, ws)):
        _assert_local(y, c, x.double() @ w.double().t(), f"y_{j}")


@pytest.mark.parametrize("T,K,Ns,dtype", [DGRAD_CASES[1], DGRAD_CASES[2], DGRAD_CASES[3]])
def test_dgrad_non_finite_inputs_stay_local(ops, T, K, Ns, dtype):
    dys, ws = _dgrad_inputs(T, K, Ns, dtype)
    clean = ops.fused_linear_dgrad(dys, ws)
    dys = [dy.clone() for dy in dys]
    ws = [w.clone() for w in ws]
    dys[1][T // 2, Ns[1] - 1] = float("nan")
    ws[2][0, K - 1] = float("inf")                          # last column of dx
    got = ops.fused_linear_dgrad(dys, ws)
    _assert_local(got, clean, _dgrad_reference(dys, ws)[0], "dx")
