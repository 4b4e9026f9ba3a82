"""GPU tests of the decoder-layer kernels (csrc/decoder_kernels.cu) away from the 8B shapes of
test_gpu_decoder_fusion.py and test_gpu_model_families.py:

  * RoPE and qk-norm RoPE with a different cos / sin row per sequence (HF's [B, S, 128] table for per-row
    `position_ids`), with HF's shared [1, S, 128] table and with a [B, S, 128] view of batch stride 0;
  * grid-stride loops that take three passes, the last one partial, and head layouts outside 32 / 8;
  * RMSNorm widths from one partly filled warp (H = 8) to the 1 024-thread maximum (H = 32 768);
  * rows holding inf, NaN, values whose fp32 sum of squares overflows, or zeros, which must stay in their own row;
  * Qwen3-0.6B- and Mistral-Nemo-shaped layers (q width != hidden size) with per-row positions and left padding,
    against fp64.

Kernels are held bit for bit to HF's formula (fed the kernel's rstd where only the order of a row sum differs), or
to an fp64 truth with HF's own error as the bar."""
import copy
import importlib

import pytest
import torch

pytestmark = pytest.mark.gpu

HD = 128
EPS = 1e-6


@pytest.fixture(scope="module")
def M(built_library):
    from sparse_matrix_tuning_b200.smt import smt
    return smt


def _grid_pass():
    """Work items one pass of a flat kernel's grid covers: `flat_grid` caps it at 16 CTAs of 256 threads per SM."""
    return 16 * torch.cuda.get_device_properties(0).multi_processor_count * 256


def _three_passes(per_unit):
    """The smallest count of units of `per_unit` work items that takes three grid passes, the last one partial."""
    n = 2 * _grid_pass() // per_unit + 1
    while (n * per_unit) % _grid_pass() == 0:
        n += 1
    assert 2 * _grid_pass() < n * per_unit < 3 * _grid_pass()
    return n


def _ulp_bf16(x):
    """Spacing of bf16 numbers at |x| (fp32 tensor)."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def _no_worse_than_hf(got, hf, truth, what=""):
    """Max error against fp64, relative to the largest |truth|, at most 1.05x HF's plus half a bf16 ulp of that
    largest value: at a few hundred elements both errors come down to a handful of final roundings."""
    scale = truth.abs().max().item()
    err, hf_err = [(t.double() - truth).abs().max().item() / scale for t in (got, hf)]
    slack = _ulp_bf16(torch.tensor(scale)).item() / 2 / scale
    assert err <= hf_err * 1.05 + slack, (what, err, hf_err)


def _rstd_near_fp64(x, rstd, eps):
    """The kernel's fp32 rstd sums the squares in another order than torch's, so it is held to torch's own fp32
    error against fp64 (twice it, plus four fp32 ulps for rsqrtf and the mean), not to torch's value."""
    x64 = x.double().reshape(rstd.numel(), -1)
    r64 = torch.rsqrt(x64.pow(2).mean(-1) + eps)
    r32 = torch.rsqrt(x.float().reshape(rstd.numel(), -1).pow(2).mean(-1) + eps).double()
    err, torch_err = [((r - r64) / r64).abs().max().item() for r in (rstd.double(), r32)]
    assert err <= 2 * torch_err + 2 ** -21, (err, torch_err)


def _same_non_finite(got, ref):
    """Same NaN and inf positions (NaN payloads and signs are not compared); returns the mask of finite elements."""
    assert torch.equal(got.isnan(), ref.isnan()) and torch.equal(got.isinf(), ref.isinf())
    assert torch.equal(got[got.isinf()], ref[ref.isinf()])
    return got.isfinite()


# ---- positions and cos / sin tables --------------------------------------------------------------------------------

def _pad(S):
    return S // 5


def _positions(B, S):
    """Position ids [B, S], a different row per sequence (B <= 4): a start at 30 000; three packed documents, whose
    positions restart at 0 twice; 0..S-1; a left-padded row as HF builds it (cumsum(mask) - 1, padding at 1)."""
    a, c, pad = S // 3, 2 * S // 3, _pad(S)
    rows = [torch.arange(S) + 30000,
            torch.cat([torch.arange(a), torch.arange(c - a), torch.arange(S - c)]),
            torch.arange(S),
            torch.cat([torch.ones(pad, dtype=torch.long), torch.arange(S - pad)])]
    assert B <= len(rows)
    return torch.stack(rows[:B]).cuda()


def _cfg(family, **kw):
    import transformers
    base = dict(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=1, num_attention_heads=4,
                num_key_value_heads=2, head_dim=HD, max_position_embeddings=256, attn_implementation="sdpa")
    base.update(kw)
    return getattr(transformers, f"{family}Config")(**base)


def _modeling(family):
    return importlib.import_module(f"transformers.models.{family.lower()}.modeling_{family.lower()}")


def _tables(family, B, S, layout):
    """cos / sin from the family's own rotary embedding: `rows` [B, S, 128] from `_positions`, `shared` the [1, S, 128]
    table of positions 0..S-1 that HF passes for a whole batch, `stride0` that table expanded to [B, S, 128]."""
    rope = getattr(_modeling(family), f"{family}RotaryEmbedding")(_cfg(family, rope_theta=5e5)).cuda()
    x = torch.zeros(1, device="cuda", dtype=torch.bfloat16)
    if layout == "rows":
        cos, sin = rope(x, _positions(B, S))
        assert all(not torch.equal(cos[i], cos[j]) for i in range(B) for j in range(i))
    else:
        cos, sin = rope(x, torch.arange(S, device="cuda")[None])
        if layout == "stride0":
            cos, sin = cos.expand(B, -1, -1), sin.expand(B, -1, -1)
            assert cos.stride(0) == 0
    return cos, sin


# (B, S, Hq, Hk, cos / sin layout); S = None: enough tokens for three grid passes
SHAPES = [(4, 64, 16, 8, "rows"), (4, 64, 16, 8, "shared"), (4, 64, 16, 8, "stride0"), (3, 40, 40, 8, "rows"),
          (4, 24, 32, 32, "rows"), (1, 1, 1, 1, "rows"), (3, 17, 3, 2, "rows"), (4, None, 40, 8, "rows")]


def _shape_id(s):
    B, S, Hq, Hk, layout = s
    return f"B{B}-S{S or 'multipass'}-{Hq}x{Hk}-{layout}"


def _qk(B, S, Hq, Hk, seed, q_scale=2.0, k_scale=0.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = (torch.randn(B, S, Hq, HD, device="cuda", generator=g) * q_scale).bfloat16()
    k = (torch.randn(B, S, Hk, HD, device="cuda", generator=g) * k_scale).bfloat16()
    return q, k, g


# ---- RoPE ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", SHAPES, ids=_shape_id)
def test_rope_bit_exact_vs_hf(built_library, shape):
    from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
    from sparse_matrix_tuning_b200 import ops
    B, S, Hq, Hk, layout = shape
    S = S or _three_passes(B * (Hq + Hk) * 8)
    q, k, g = _qk(B, S, Hq, Hk, seed=S * 131 + Hq, q_scale=1.0, k_scale=1.0)
    cos, sin = _tables("Llama", B, S, layout)
    qt, kt = q.transpose(1, 2).requires_grad_(True), k.transpose(1, 2).requires_grad_(True)
    q_ref, k_ref = apply_rotary_pos_emb(qt, kt, cos, sin)
    q_got, k_got = ops.rope_forward(q, k, cos, sin)
    assert torch.equal(q_got.transpose(1, 2), q_ref) and torch.equal(k_got.transpose(1, 2), k_ref)
    assert all(torch.equal(a, b) for a, b in zip(ops.rope_forward(q, k, cos, sin), (q_got, k_got)))
    dq_out = torch.randn(q.shape, device="cuda", generator=g).bfloat16()
    dk_out = torch.randn(k.shape, device="cuda", generator=g).bfloat16()
    dq_ref, dk_ref = torch.autograd.grad((q_ref, k_ref), (qt, kt), (dq_out.transpose(1, 2), dk_out.transpose(1, 2)))
    dq, dk = ops.rope_backward(dq_out, dk_out, cos, sin)
    assert torch.equal(dq.transpose(1, 2), dq_ref) and torch.equal(dk.transpose(1, 2), dk_ref)


# ---- qk-norm RoPE ----------------------------------------------------------------------------------------------------

def _hf_norm(x, w, eps, rstd=None):
    """Qwen3RMSNorm's arithmetic; with `rstd` given, that value instead of its own."""
    xf = x.float()
    if rstd is None:
        rstd = torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)
    return w * (xf * rstd).to(x.dtype)


def _hf_qk(q, k, wq, wk, eps_q, eps_k, cos, sin, rq=None, rk=None):
    """HF's q_norm / k_norm + apply_rotary_pos_emb, in the kernel's [B, S, H, 128] layout."""
    from transformers.models.qwen3.modeling_qwen3 import apply_rotary_pos_emb
    B, S, Hq, Hk = *q.shape[:3], k.shape[2]
    rq = None if rq is None else rq.view(B, S, Hq, 1)
    rk = None if rk is None else rk.view(B, S, Hk, 1)
    qo, ko = apply_rotary_pos_emb(_hf_norm(q, wq, eps_q, rq).transpose(1, 2), _hf_norm(k, wk, eps_k, rk).transpose(1, 2),
                                  cos, sin)
    return qo.transpose(1, 2), ko.transpose(1, 2)


def _norm_weights(g):
    return [(1 + 0.1 * torch.randn(HD, device="cuda", generator=g)).bfloat16() for _ in range(2)]


def _qk_grads64(q, k, wq, wk, eps_q, eps_k, cos, sin, dq_o, dk_o):
    """fp64 truth and HF's bf16 autograd of q_norm / k_norm + RoPE."""
    from transformers.models.qwen3.modeling_qwen3 import apply_rotary_pos_emb
    q64, k64 = q.double().requires_grad_(True), k.double().requires_grad_(True)

    def norm64(x, w, eps):
        return w.double() * x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + eps)
    r64 = apply_rotary_pos_emb(norm64(q64, wq, eps_q).transpose(1, 2), norm64(k64, wk, eps_k).transpose(1, 2),
                               cos.double(), sin.double())
    truth = torch.autograd.grad(r64, (q64, k64), (dq_o.double().transpose(1, 2), dk_o.double().transpose(1, 2)))
    qh, kh = q.clone().requires_grad_(True), k.clone().requires_grad_(True)
    hf = torch.autograd.grad(_hf_qk(qh, kh, wq, wk, eps_q, eps_k, cos, sin), (qh, kh), (dq_o, dk_o))
    return truth, hf


@pytest.mark.parametrize("shape", SHAPES, ids=_shape_id)
def test_qk_norm_rope_against_hf_and_fp64(built_library, shape):
    from sparse_matrix_tuning_b200 import ops
    B, S, Hq, Hk, layout = shape
    S = S or _three_passes(B * (Hq + Hk) * 8)
    q, k, g = _qk(B, S, Hq, Hk, seed=S * 137 + Hq)
    wq, wk = _norm_weights(g)
    cos, sin = _tables("Qwen3", B, S, layout)
    qo, ko, rq, rk = ops.qk_norm_rope_forward(q, k, wq, wk, EPS, EPS, cos, sin)
    _rstd_near_fp64(q, rq, EPS)
    _rstd_near_fp64(k, rk, EPS)
    q_own, k_own = _hf_qk(q, k, wq, wk, EPS, EPS, cos, sin, rq, rk)
    assert torch.equal(qo, q_own) and torch.equal(ko, k_own)
    again = ops.qk_norm_rope_forward(q, k, wq, wk, EPS, EPS, cos, sin)
    assert all(torch.equal(a, b) for a, b in zip(again, (qo, ko, rq, rk)))
    dq_o = torch.randn(q.shape, device="cuda", generator=g).bfloat16()
    dk_o = torch.randn(k.shape, device="cuda", generator=g).bfloat16()
    truth, hf = _qk_grads64(q, k, wq, wk, EPS, EPS, cos, sin, dq_o, dk_o)
    got = ops.qk_norm_rope_backward(q, k, wq, wk, rq, rk, cos, sin, dq_o, dk_o)
    for what, t, h, x in zip(("dq", "dk"), truth, hf, got):
        _no_worse_than_hf(x, h, t, what)


def test_qk_norm_rope_applies_eps_q_to_q_and_eps_k_to_k(built_library):
    """At |x| ~ 1e-3, mean(x^2) ~ 1e-6: an eps of 1e-2 dominates the norm, so q and k with swapped eps differ."""
    from sparse_matrix_tuning_b200 import ops
    B, S, Hq, Hk = 2, 16, 4, 2
    eps_q, eps_k = 1e-6, 1e-2
    q, k, g = _qk(B, S, Hq, Hk, seed=11, q_scale=1e-3, k_scale=1e-3)
    wq, wk = _norm_weights(g)
    cos, sin = _tables("Qwen3", B, S, "rows")
    qo, ko, rq, rk = ops.qk_norm_rope_forward(q, k, wq, wk, eps_q, eps_k, cos, sin)
    _rstd_near_fp64(q, rq, eps_q)
    _rstd_near_fp64(k, rk, eps_k)
    q_own, k_own = _hf_qk(q, k, wq, wk, eps_q, eps_k, cos, sin, rq, rk)
    assert torch.equal(qo, q_own) and torch.equal(ko, k_own)
    q_hf, k_hf = _hf_qk(q, k, wq, wk, eps_q, eps_k, cos, sin)
    q_sw, k_sw = _hf_qk(q, k, wq, wk, eps_k, eps_q, cos, sin)
    for got, ref, swapped in ((qo, q_hf, q_sw), (ko, k_hf, k_sw)):
        err, err_sw = [(got.float() - r.float()).abs().max().item() for r in (ref, swapped)]
        assert err <= 0.02 * ref.float().abs().max().item() < err_sw, (err, err_sw)
    dq_o = torch.randn(q.shape, device="cuda", generator=g).bfloat16()
    dk_o = torch.randn(k.shape, device="cuda", generator=g).bfloat16()
    truth, hf = _qk_grads64(q, k, wq, wk, eps_q, eps_k, cos, sin, dq_o, dk_o)
    got = ops.qk_norm_rope_backward(q, k, wq, wk, rq, rk, cos, sin, dq_o, dk_o)
    for what, t, h, x in zip(("dq", "dk"), truth, hf, got):
        _no_worse_than_hf(x, h, t, what)


# ---- non-finite and saturating rows -----------------------------------------------------------------------------------

_KINDS = ("inf", "nan", "huge", "zero")


def _poison(x2d, rows, g):
    """Writes each kind of bad row into `x2d` [rows, width]: one +-inf element, one NaN element, a row of bf16 values
    near +-3e38 (the fp32 sum of squares overflows), an all-zero row."""
    n = x2d.shape[1]
    for kind, rs in zip(_KINDS, rows):
        for r in rs:
            col = (r * 37) % n
            if kind == "inf":
                x2d[r, col] = float("inf") if r % 2 else float("-inf")
            elif kind == "nan":
                x2d[r, col] = float("nan")
            elif kind == "huge":
                sign = torch.randint(0, 2, (n,), device="cuda", generator=g) * 2 - 1
                x2d[r] = (3.0e38 * sign).to(x2d.dtype)
                assert x2d[r].isfinite().all() and torch.isinf(x2d[r].float().pow(2).sum())
            else:
                x2d[r] = 0


def _warp_rows(n_rows, base):
    """Rows of each kind such that every kind sits at each of the four head-row slots of a warp (global row index
    `base + r` mod 4 = 0..3): the kernel's 8-lane shuffles of four rows share one warp."""
    rows = [[4 * (4 * i + j + 1) + (i + j - base) % 4 for j in range(4)] for i in range(len(_KINDS))]
    assert max(max(r) for r in rows) < n_rows
    assert all(sorted((base + r) % 4 for r in rs) == [0, 1, 2, 3] for rs in rows)
    return rows


def _bad_row_mask(n_rows, rows):
    m = torch.zeros(n_rows, dtype=torch.bool, device="cuda")
    m[[r for rs in rows for r in rs]] = True
    return m


def test_qk_norm_rope_keeps_non_finite_rows_to_themselves(built_library):
    from sparse_matrix_tuning_b200 import ops
    B, S, Hq, Hk = 3, 9, 5, 3              # 135 q rows: one warp holds the last q rows and the first k rows
    q, k, g = _qk(B, S, Hq, Hk, seed=12)
    wq, wk = _norm_weights(g)
    cos, sin = _tables("Qwen3", B, S, "rows")
    nq, nk = B * S * Hq, B * S * Hk
    rows_q, rows_k = _warp_rows(nq, 0), _warp_rows(nk, nq)
    bq, bk = q.clone(), k.clone()
    _poison(bq.view(nq, HD), rows_q, g)
    _poison(bk.view(nk, HD), rows_k, g)
    bad_q, bad_k = _bad_row_mask(nq, rows_q), _bad_row_mask(nk, rows_k)
    clean = ops.qk_norm_rope_forward(q, k, wq, wk, EPS, EPS, cos, sin)
    qo, ko, rq, rk = ops.qk_norm_rope_forward(bq, bk, wq, wk, EPS, EPS, cos, sin)
    q_hf, k_hf = _hf_qk(bq, bk, wq, wk, EPS, EPS, cos, sin)
    q_own, k_own = _hf_qk(bq, bk, wq, wk, EPS, EPS, cos, sin, rq, rk)
    for got, hf, own, c, r, bad, n in ((qo, q_hf, q_own, clean[0], rq, bad_q, nq), (ko, k_hf, k_own, clean[1], rk, bad_k, nk)):
        _same_non_finite(got, hf)
        fin = _same_non_finite(got, own)
        assert torch.equal(got[fin], own[fin])
        assert torch.equal(got.view(n, HD)[~bad], c.view(n, HD)[~bad])
    assert torch.equal(rq[~bad_q], clean[2][~bad_q]) and torch.equal(rk[~bad_k], clean[3][~bad_k])

    dq_o = torch.randn(q.shape, device="cuda", generator=g).bfloat16()
    dk_o = torch.randn(k.shape, device="cuda", generator=g).bfloat16()
    clean_d = ops.qk_norm_rope_backward(q, k, wq, wk, clean[2], clean[3], cos, sin, dq_o, dk_o)
    got = ops.qk_norm_rope_backward(bq, bk, wq, wk, rq, rk, cos, sin, dq_o, dk_o)
    truth, hf = _qk_grads64(bq, bk, wq, wk, EPS, EPS, cos, sin, dq_o, dk_o)
    for x, h, t, c, rows, n in zip(got, hf, truth, clean_d, (rows_q, rows_k), (nq, nk)):
        _bad_rows_backward(x.view(n, HD), h.reshape(n, HD), t.reshape(n, HD), c.view(n, HD), rows)


def _bad_rows_backward(got, hf, truth, clean, rows):
    """Input gradients [rows, width] of a norm whose input holds `_poison`'s rows.  inf / NaN rows take HF's
    non-finite pattern (all NaN); zero rows are within HF's error of fp64; every clean row is bit-identical to a clean
    run.  On a huge row HF's autograd gives NaN (its pow backward forms 2x, which overflows fp32) while fp64 gives
    values below 1e-37 (rstd ~ 1 / 3e38): the kernel's rstd of 0 must give exact zeros there."""
    inf, nan, huge, zero = rows
    _same_non_finite(got[inf + nan], hf[inf + nan])
    assert (truth[huge].abs() < 1e-37).all() and (got[huge] == 0).all()
    _no_worse_than_hf(got[zero], hf[zero], truth[zero], "zero rows")
    bad = _bad_row_mask(got.shape[0], rows)
    assert torch.equal(got[~bad], clean[~bad])


# ---- RMSNorm ---------------------------------------------------------------------------------------------------------

# one partly filled warp (8), a partial last vector pass (520, 2560, 5120), a last thread holding fewer vectors than the
# others (1032: 129 vectors over 64 threads), whole passes (1024, 8192) and the 1 024-thread maximum (32 768)
WIDTHS = [8, 520, 1024, 1032, 2560, 5120, 8192, 32768]


def _norm_inputs(T, H, seed, residual):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(T, H, device="cuda", generator=g).bfloat16()
    res = torch.randn(T, H, device="cuda", generator=g).bfloat16() if residual else None
    w = (1 + 0.1 * torch.randn(H, device="cuda", generator=g)).bfloat16()
    return a, res, w, g


def _check_norm_forward(a, res, w, eps):
    from sparse_matrix_tuning_b200 import ops
    y, rstd, h = ops.rmsnorm_forward(a, w, eps, res=res)
    x = a if res is None else res + a
    if res is not None:
        assert torch.equal(h, x)
    if x.shape[0]:
        _rstd_near_fp64(x, rstd, eps)
    assert torch.equal(y, w * (x.float() * rstd[:, None]).bfloat16())      # HF's formula fed the kernel's rstd
    y2, rstd2, h2 = ops.rmsnorm_forward(a, w, eps, res=res)
    assert torch.equal(y, y2) and torch.equal(rstd, rstd2) and (h is None or torch.equal(h, h2))
    return y, rstd, x


def _norm_grads64(x, w, eps, dy, dres):
    """fp64 truth and HF's bf16 autograd of the norm's input gradient, plus `dres`."""
    x64 = x.double().requires_grad_(True)
    y64 = w.double() * (x64 * torch.rsqrt(x64.pow(2).mean(-1, keepdim=True) + eps))
    truth = torch.autograd.grad(y64, x64, dy.double())[0] + (0 if dres is None else dres.double())
    xh = x.clone().requires_grad_(True)
    hf = torch.autograd.grad(w * (xh.float() * torch.rsqrt(xh.float().pow(2).mean(-1, keepdim=True) + eps))
                             .to(x.dtype), xh, dy)[0]
    if dres is not None:
        hf = hf + dres                                                       # autograd's bf16 add at the fork
    return truth, hf


def _check_norm_backward(x, w, rstd, eps, dy, dres):
    from sparse_matrix_tuning_b200 import ops
    truth, hf = _norm_grads64(x, w, eps, dy, dres)
    got = ops.rmsnorm_backward(x, w, rstd, dy, dres)
    _no_worse_than_hf(got, hf, truth)
    assert torch.equal(got, ops.rmsnorm_backward(x, w, rstd, dy, dres))


@pytest.mark.parametrize("residual", [False, True], ids=["plain", "residual"])
@pytest.mark.parametrize("H", WIDTHS)
def test_rmsnorm_at_width(built_library, H, residual):
    eps = 1e-5
    a, res, w, g = _norm_inputs(37, H, seed=H + residual, residual=residual)
    _y, rstd, x = _check_norm_forward(a, res, w, eps)
    dy = torch.randn(x.shape, device="cuda", generator=g).bfloat16()
    dres = torch.randn(x.shape, device="cuda", generator=g).bfloat16() if residual else None
    _check_norm_backward(x, w, rstd, eps, dy, dres)


@pytest.mark.parametrize("T", [0, 1])
def test_rmsnorm_at_zero_and_one_row(built_library, T):
    from sparse_matrix_tuning_b200 import ops
    for H in (8, 2560):
        a, res, w, g = _norm_inputs(T, H, seed=T, residual=True)
        for r in (None, res):
            y, rstd, x = _check_norm_forward(a, r, w, 1e-6)
            assert y.shape == (T, H) and rstd.shape == (T,)
            dy = torch.randn(x.shape, device="cuda", generator=g).bfloat16()
            if T:
                _check_norm_backward(x, w, rstd, 1e-6, dy, r)
            else:
                assert ops.rmsnorm_backward(x, w, rstd, dy, r).shape == (0, H)


@pytest.mark.parametrize("H", [8, 2560])
def test_rmsnorm_keeps_non_finite_rows_to_themselves(built_library, H):
    from sparse_matrix_tuning_b200 import ops
    eps = 1e-5
    T = 21
    rows = [[1, 14], [4], [7, 20], [10]]
    a, _res, w, g = _norm_inputs(T, H, seed=H + 5, residual=False)
    x = a.clone()
    _poison(x, rows, g)
    bad = _bad_row_mask(T, rows)
    y_c, r_c, _ = ops.rmsnorm_forward(a, w, eps)
    y, rstd, _ = ops.rmsnorm_forward(x, w, eps)
    xf = x.float()
    hf = w * (xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)).bfloat16()
    own = w * (xf * rstd[:, None]).bfloat16()
    _same_non_finite(y, hf)
    fin = _same_non_finite(y, own)
    assert torch.equal(y[fin], own[fin])
    assert torch.equal(y[~bad], y_c[~bad]) and torch.equal(rstd[~bad], r_c[~bad])

    dy = torch.randn(T, H, device="cuda", generator=g).bfloat16()
    dres = torch.randn(T, H, device="cuda", generator=g).bfloat16()
    for d in (None, dres):
        got = ops.rmsnorm_backward(x, w, rstd, dy, d)
        c = ops.rmsnorm_backward(a, w, r_c, dy, d)
        truth, hf = _norm_grads64(x, w, eps, dy, d)
        if d is not None:                  # on a huge row only the residual stream's gradient reaches x, exactly
            huge = rows[_KINDS.index("huge")]
            assert torch.equal(got[huge], d[huge])
            got, truth = got.clone(), truth.clone()
            got[huge], truth[huge] = 0, truth[huge] - d[huge].double()
        _bad_rows_backward(got, hf, truth, c, rows)


def test_norm_width_limit_selects_the_native_path(built_library, monkeypatch):
    """`_MAX_NORM_WIDTH` (the C limit, 32 768) and the next multiple of 8: the first runs the kernel, the second
    the class's own forward."""
    from transformers.models.llama.modeling_llama import LlamaRMSNorm
    from sparse_matrix_tuning_b200 import decoder_fusion as D, ops
    calls = []
    fwd = ops.rmsnorm_forward
    monkeypatch.setattr(ops, "rmsnorm_forward", lambda *a, **k: calls.append(1) or fwd(*a, **k))
    for H, native in ((D._MAX_NORM_WIDTH, True), (D._MAX_NORM_WIDTH + 8, False)):
        norm = LlamaRMSNorm(H, eps=1e-5).cuda().bfloat16()
        norm.weight.requires_grad_(False)
        x = torch.randn(3, H, device="cuda").bfloat16()
        ref = norm(x)
        calls.clear()
        assert D.install_norm(norm)
        got = norm(x)
        assert len(calls) == native
        if native:
            assert ((got.float() - ref.float()).abs() <= _ulp_bf16(ref.float())).all()
        else:
            assert torch.equal(got, ref)


# ---- SwiGLU ----------------------------------------------------------------------------------------------------------

def _swiglu_check(g, u, dh):
    """Forward bit for bit with torch's `silu(g) * u` on finite values and on the NaN / inf pattern; backward
    within one bf16 ulp of autograd with the same pattern; a second forward is bit-identical."""
    from sparse_matrix_tuning_b200 import ops
    gr, ur = g.clone().requires_grad_(True), u.clone().requires_grad_(True)
    h_ref = torch.nn.functional.silu(gr) * ur
    h = ops.swiglu_forward(g, u)
    fin = _same_non_finite(h, h_ref)
    assert torch.equal(h[fin], h_ref[fin])
    again = ops.swiglu_forward(g, u)
    assert torch.equal(h.isnan(), again.isnan()) and torch.equal(h.nan_to_num(), again.nan_to_num())
    refs = torch.autograd.grad(h_ref, (gr, ur), dh)
    for got, ref in zip(ops.swiglu_backward(g, u, dh), refs):
        fin = _same_non_finite(got, ref)
        diff = (got[fin].float() - ref[fin].float()).abs()
        assert (diff <= _ulp_bf16(ref[fin].float())).all(), diff.max().item()


@pytest.mark.parametrize("n", ["8", "1000x8", "multipass"])
def test_swiglu_at_length(built_library, n):
    """n = 8 (one vector), 1 000 vectors (not a multiple of the 256-thread block), and a length whose vectors take
    three grid passes, the last one partial and not a multiple of 256."""
    nvec = {"8": 1, "1000x8": 1000}.get(n, 2 * _grid_pass() + 37)
    g = torch.Generator(device="cuda").manual_seed(nvec)
    x = [(torch.randn(nvec * 8, device="cuda", generator=g) * s).bfloat16() for s in (3.0, 1.0, 1.0)]
    _swiglu_check(*x)


def test_swiglu_at_non_finite_and_saturating_gates(built_library):
    """g over inf, NaN, the expf overflow boundary of silu (|g| 88 .. 104) and bf16 subnormals, each paired with
    u in {0, +-inf} and ordinary values."""
    sub = [2.0 ** -133, 2.0 ** -127, -(2.0 ** -130), 3 * 2.0 ** -133]
    edge = [88.0, 88.5, 88.75, 89.0, 90.0, 96.0, 100.0, 104.0]
    gv = [float("inf"), float("-inf"), float("nan"), 0.0, 1.0, -2.5] + edge + [-e for e in edge] + sub
    uv = [0.0, float("inf"), float("-inf"), 1.5, -0.75, 3.0]
    gg, uu = torch.meshgrid(torch.tensor(gv), torch.tensor(uv), indexing="ij")
    n = -(-gg.numel() // 8) * 8
    g = torch.zeros(n, dtype=torch.bfloat16, device="cuda")
    u = torch.ones(n, dtype=torch.bfloat16, device="cuda")
    g[:gg.numel()], u[:uu.numel()] = gg.reshape(-1).bfloat16(), uu.reshape(-1).bfloat16()
    assert ((g != 0) & (g.float().abs() < 2.0 ** -126)).sum() == len(sub) * len(uv)   # subnormals survived the cast
    dh = torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(13)).bfloat16()
    _swiglu_check(g, u, dh)


# ---- decoder layers whose q width is not the hidden size, against fp64 -------------------------------------------------

def _mask(B, S, pad):
    """Causal bool mask [B, 1, S, S] with the first `pad` tokens of the last sequence left padding; a padded query
    sees only itself, so no row is empty."""
    keep = torch.ones(B, S, dtype=torch.bool, device="cuda")
    keep[-1, :pad] = False
    causal = torch.ones(S, S, dtype=torch.bool, device="cuda").tril()
    m = causal[None] & keep[:, None, :]
    m |= torch.eye(S, dtype=torch.bool, device="cuda")[None]
    return m[:, None], keep


@pytest.mark.parametrize("family,widths,sel", [
    ("Qwen3", dict(hidden_size=1024, num_attention_heads=16, num_key_value_heads=8, intermediate_size=3072),
     {"q_proj": [(0, 1), (7, 3)], "k_proj": [(1, 2), (3, 0)], "v_proj": [(2, 3)]}),
    ("Mistral", dict(hidden_size=5120, num_attention_heads=32, num_key_value_heads=8, intermediate_size=14336,
                     sliding_window=None),
     {"q_proj": [(0, 1), (5, 19), (15, 15)], "k_proj": [(1, 2), (3, 0)], "v_proj": [(2, 7)]}),
], ids=["qwen3_0.6b", "mistral_nemo"])
def test_decoder_layer_with_padding_and_per_row_positions_against_fp64(M, family, widths, sel):
    """Output, dx and compact block gradients of the fused layer (SMT q/k/v blocks, non-reentrant checkpointing) are
    no further from fp64 than the HF layer's (x 1.25 + 1e-4), on the tokens that are not padding."""
    from torch.utils.checkpoint import checkpoint
    mod = _modeling(family)
    cfg = _cfg(family, head_dim=HD, rms_norm_eps=EPS, rope_theta=1e6, **widths)
    assert cfg.num_attention_heads * HD != cfg.hidden_size
    torch.manual_seed(5)
    base = getattr(mod, f"{family}DecoderLayer")(cfg, 0).cuda()
    with torch.no_grad():
        for n, p in base.named_parameters():
            p.copy_(1 + 0.1 * torch.randn_like(p) if "norm" in n else torch.randn_like(p) * 0.02)
    B, S = 4, 128
    H = cfg.hidden_size
    x = torch.randn(B, S, H, device="cuda")
    pos = _positions(B, S)
    mask, keep = _mask(B, S, _pad(S))
    dout = torch.randn(B, S, H, device="cuda") * keep[..., None]
    rope = getattr(mod, f"{family}RotaryEmbedding")(cfg).cuda()

    def run(dtype, fuse):
        layer = copy.deepcopy(base).to(dtype)
        for p in layer.parameters():
            p.requires_grad_(False)
        attn = layer.self_attn
        if dtype == torch.float64:
            for name in sel:
                getattr(attn, name).weight.requires_grad_(True)
        else:
            for name, idx in sel.items():
                setattr(attn, name, M.LinearLayer_MatrixSparsity(getattr(attn, name).weight, index_list=idx))
            if fuse:
                assert M.fuse_qkv_projections(layer) == 1 and "forward" in layer.__dict__
        pe = rope(x.to(dtype), pos)
        xin = x.to(dtype).requires_grad_(True)
        out = checkpoint(lambda t: layer(t, attention_mask=mask, position_embeddings=pe, position_ids=pos), xin,
                         use_reentrant=False)
        out.backward(dout.to(dtype))
        if dtype == torch.float64:
            blocks = [getattr(attn, n).weight.grad[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256]
                      for n, idx in sel.items() for r, c in idx]
        else:
            blocks = [getattr(attn, n).selected_weight.grad.view(-1, 256, 256)[i]
                      for n, idx in sel.items() for i in range(len(idx))]
        return out.detach()[keep].double(), xin.grad[keep].double(), torch.stack(blocks).double()

    truth = run(torch.float64, False)
    hf = run(torch.bfloat16, False)
    fused = run(torch.bfloat16, True)
    for what, t, h, f in zip(("output", "dx", "block grads"), truth, hf, fused):
        assert torch.isfinite(f).all(), what
        scale = t.abs().max().item()
        e_hf, e_f = (h - t).abs().max().item() / scale, (f - t).abs().max().item() / scale
        assert e_f <= e_hf * 1.25 + 1e-4, (what, e_f, e_hf)
