"""GPU tests of the fused lm_head + causal-LM cross-entropy: the row kernel (csrc/loss_kernels.cu), the chunked
`LinearCrossEntropyFn` at LLaMA-3-8B widths against an fp64 truth and against transformers' loss, and the
`LlamaForCausalLM` override installed by `fuse_causal_lm_loss`, with its fallbacks."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu

HID, VOCAB = 4096, 128256          # LLaMA-3-8B widths


@pytest.fixture(scope="module")
def M(built_library):
    from sparse_matrix_tuning_b200.smt import smt
    return smt


@pytest.fixture
def ce_calls(monkeypatch, built_library):
    """Counts calls of `ops.cross_entropy_rows`."""
    from sparse_matrix_tuning_b200 import ops
    calls = {"n": 0}
    fn = ops.cross_entropy_rows

    def wrapped(*a, **k):
        calls["n"] += 1
        return fn(*a, **k)
    monkeypatch.setattr(ops, "cross_entropy_rows", wrapped)
    return calls


def _ulp_bf16(x):
    """Spacing of bf16 numbers at |x| (fp32 tensor)."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def _hf_grad(logits, labels, reduction="mean"):
    """transformers' loss on `.float()` logits, its gradient through autograd, `.bfloat16()`."""
    xf = logits.float().requires_grad_(True)
    loss = torch.nn.functional.cross_entropy(xf, labels, ignore_index=-100, reduction=reduction)
    loss.backward()
    return loss.detach(), xf.grad.bfloat16()


# ---- the row kernel --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("V", [32000, VOCAB])
def test_kernel_loss_and_gradient_against_fp64_and_hf(built_library, V):
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(0)
    T = 96
    x = (torch.randn(T, V, device="cuda") * 3).bfloat16()
    y = torch.randint(0, V, (T,), device="cuda")
    y[::7] = -100
    n_valid = (y != -100).sum()
    scale = (1.0 / n_valid.float()).reshape(1)
    g = x.clone()
    loss_rows = ops.cross_entropy_rows(g, y, scale, -100)
    x64 = x.double()
    valid = y != -100
    truth = torch.logsumexp(x64, -1) - x64.gather(1, y.clamp_min(0)[:, None])[:, 0]
    truth[~valid] = 0
    assert torch.allclose(loss_rows.double(), truth, rtol=1e-5, atol=0), (loss_rows.double() - truth).abs().max()
    assert (loss_rows[~valid] == 0).all()
    hf_loss, hf_g = _hf_grad(x, y)
    assert torch.allclose(loss_rows.sum() / n_valid, hf_loss, rtol=1e-5)
    diff = (g.float() - hf_g.float()).abs()
    assert (diff <= _ulp_bf16(hf_g.float())).all(), diff.max().item()
    assert (g[~valid] == 0).all()
    # deterministic
    g2 = x.clone()
    assert torch.equal(ops.cross_entropy_rows(g2, y, scale, -100), loss_rows) and torch.equal(g2, g)


def test_kernel_out_of_range_label_gives_nan_for_that_row_only(built_library):
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(1)
    T, V = 16, 32000
    x = torch.randn(T, V, device="cuda").bfloat16()
    y = torch.randint(0, V, (T,), device="cuda")
    scale = torch.full((1,), 1.0 / T, device="cuda")
    g_ref = x.clone()
    l_ref = ops.cross_entropy_rows(g_ref, y, scale, -100)
    for bad in (V, V + 1000, -5):
        yb = y.clone()
        yb[3] = bad
        g = x.clone()
        loss = ops.cross_entropy_rows(g, yb, scale, -100)
        torch.cuda.synchronize()
        assert torch.isnan(loss[3]) and torch.isnan(g[3].float()).all()
        others = torch.arange(T, device="cuda") != 3
        assert torch.equal(loss[others], l_ref[others]) and torch.equal(g[others], g_ref[others])


def test_kernel_all_labels_ignored_matches_torch(built_library):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    torch.manual_seed(2)
    T, K, V = 256, 256, 32000
    h = (torch.randn(T, K, device="cuda")).bfloat16().requires_grad_(True)
    w = (torch.randn(V, K, device="cuda") * 0.05).bfloat16()
    labels = torch.full((1, T), -100, device="cuda")
    loss = D.causal_lm_loss(h, w, labels)
    loss.backward()
    hf_loss, _ = _hf_grad(h.detach() @ w.T, labels.reshape(-1))
    assert torch.isnan(loss) and torch.isnan(hf_loss)
    assert (h.grad == 0).all()


# ---- lm_head + loss at LLaMA-3-8B widths -----------------------------------------------------------------------------

def _op_inputs(T, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.randn(T, HID, device="cuda", generator=g).bfloat16()
    w = (torch.randn(VOCAB, HID, device="cuda", generator=g) * 0.02).bfloat16()
    y = torch.randint(0, VOCAB, (T,), device="cuda", generator=g)
    y[torch.rand(T, device="cuda", generator=g) < 0.2] = -100
    return h, w, y


def _fused(h, w, y, num_items=None):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    hg = h.clone().requires_grad_(True)
    loss = D.causal_lm_loss(hg, w, y[None], shift_labels=y[None], num_items_in_batch=num_items)
    loss.backward()
    return loss.detach(), hg.grad


def _hf(h, w, y, num_items=None):
    from transformers.loss.loss_utils import ForCausalLMLoss
    hg = h.clone().requires_grad_(True)
    logits = torch.nn.functional.linear(hg, w)
    loss = ForCausalLMLoss(logits[None], None, VOCAB, num_items_in_batch=num_items, shift_labels=y[None])
    loss.backward()
    return loss.detach(), hg.grad


@pytest.mark.parametrize("num_items", [None, 1234])
def test_linear_cross_entropy_no_worse_than_hf_against_fp64(built_library, monkeypatch, num_items):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    T = 2048
    h, w, y = _op_inputs(T)
    h64, w64 = h.double(), w.double()
    logits64 = h64 @ w64.T
    valid = y != -100
    lse = torch.logsumexp(logits64, -1)
    rows = (lse - logits64.gather(1, y.clamp_min(0)[:, None])[:, 0]) * valid
    denom = float(valid.sum().item() if num_items is None else num_items)
    loss64 = rows.sum() / denom
    p = torch.softmax(logits64, -1)
    p[torch.arange(T, device="cuda"), y.clamp_min(0)] -= 1
    dh64 = ((p * valid[:, None]) / denom) @ w64
    del logits64, p
    nums = None if num_items is None else torch.tensor(num_items, device="cuda")
    hf_loss, hf_dh = _hf(h, w, y, nums)
    loss, dh = _fused(h, w, y, nums)
    e_hf, e = (hf_loss.double() - loss64).abs().item(), (loss.double() - loss64).abs().item()
    assert e <= 1.5 * e_hf + 1e-4 * loss64.abs().item(), (e, e_hf)
    d_hf, d = (hf_dh.double() - dh64).abs().max().item(), (dh.double() - dh64).abs().max().item()
    assert d <= 1.5 * d_hf, (d, d_hf)
    # bit-identical across calls and across chunk sizes
    loss2, dh2 = _fused(h, w, y, nums)
    assert torch.equal(loss, loss2) and torch.equal(dh, dh2)
    monkeypatch.setattr(D, "_CE_CHUNK_ROWS", 256)
    loss3, dh3 = _fused(h, w, y, nums)
    assert torch.equal(loss, loss3) and torch.equal(dh, dh3)


def test_linear_cross_entropy_ragged_last_chunk_and_no_tokens(built_library, monkeypatch):
    """600 tokens (not a multiple of 256) in chunks of 256: the last chunk has 88 rows.  Same bits as one chunk, no
    worse than HF against fp64.  No tokens at all: a NaN loss (0 / 0, as torch gives) and an empty gradient."""
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    T, K, V = 600, 512, 32000
    g = torch.Generator(device="cuda").manual_seed(8)
    h = torch.randn(T, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(V, K, device="cuda", generator=g) * 0.05).bfloat16()
    y = torch.randint(0, V, (T,), device="cuda", generator=g)
    y[::5] = -100
    whole = _fused(h, w, y)
    monkeypatch.setattr(D, "_CE_CHUNK_ROWS", 256)
    loss, dh = _fused(h, w, y)
    assert torch.equal(loss, whole[0]) and torch.equal(dh, whole[1])
    hg = h.double().requires_grad_(True)
    loss64 = torch.nn.functional.cross_entropy(hg @ w.double().T, y, ignore_index=-100)
    dh64, = torch.autograd.grad(loss64, hg)
    hh = h.clone().requires_grad_(True)
    hf_loss = torch.nn.functional.cross_entropy(torch.nn.functional.linear(hh, w).float(), y, ignore_index=-100)
    hf_loss.backward()
    hf_dh = hh.grad
    assert (loss.double() - loss64).abs() <= 1.5 * (hf_loss.double() - loss64).abs() + 1e-4 * loss64.abs()
    assert (dh.double() - dh64).abs().max() <= 1.5 * (hf_dh.double() - dh64).abs().max()
    empty = torch.empty(0, K, device="cuda", dtype=torch.bfloat16).requires_grad_(True)
    loss0 = D.causal_lm_loss(empty, w, y[:0][None], shift_labels=y[:0][None])
    loss0.backward()
    assert torch.isnan(loss0) and empty.grad.shape == (0, K)


def test_linear_cross_entropy_peak_memory_a_quarter_of_hf(built_library):
    T = 8192
    h, w, y = _op_inputs(T, seed=4)
    peaks = {}
    for name, fn in (("fused", _fused), ("hf", _hf), ("fused", _fused)):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = fn(h, w, y)
        torch.cuda.synchronize()
        peaks[name] = torch.cuda.max_memory_allocated() - base
        del out
    assert peaks["fused"] <= peaks["hf"] / 4, peaks


# ---- the LlamaForCausalLM override -----------------------------------------------------------------------------------

def _tiny_cfg(**kw):
    from transformers import LlamaConfig
    base = dict(vocab_size=32000, hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
                num_key_value_heads=2, head_dim=128, max_position_embeddings=256, attn_implementation="sdpa")
    base.update(kw)
    return LlamaConfig(**base)


def _batch(gen, vocab=32000):
    ids = torch.randint(0, vocab, (2, 128), generator=gen)
    labels = ids.clone()
    labels[:, :40] = -100                                   # prompt tokens
    return ids.cuda(), labels.cuda()


def _train(M, fuse_loss, fuse_qkv, steps=5, lr=1e-3):
    from transformers import LlamaForCausalLM
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda().bfloat16()
    sel = {("q_proj", 0): [(0, 1), (1, 0)], ("k_proj", 0): [(0, 0)], ("v_proj", 1): [(0, 1)], ("q_proj", 1): [(1, 1)]}
    M.freeze_unselected_matrix_layer(model, {}, sel)
    M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    assert not model.lm_head.weight.requires_grad
    model.train()
    if fuse_qkv:
        model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
        model.enable_input_require_grads()
        assert M.fuse_qkv_projections(model) == 2
    if fuse_loss:
        assert M.fuse_causal_lm_loss(model)
    opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, lr), betas=(0.9, 0.95), max_grad_norm=1.0)
    params = [p for g in opt.param_groups for p in g["params"]]
    M.set_grouped_backward(True)
    try:
        gen = torch.Generator().manual_seed(1)
        losses, first_grads = [], None
        for _ in range(steps):
            ids, labels = _batch(gen)
            opt.zero_grad()
            out = model(input_ids=ids, labels=labels, use_cache=False)
            assert (out.logits is None) == fuse_loss
            out.loss.backward()
            if first_grads is None:
                M.flush_block_grads()
                first_grads = [p.grad.detach().float().clone() for p in params]
            opt.step()
            losses.append(out.loss.item())
        return losses, first_grads
    finally:
        M.set_grouped_backward(False)
        M.unfuse_qkv_projections(model)


@pytest.mark.parametrize("fuse_qkv", [False, True])
def test_tiny_llama_smt_training_fused_loss_matches_hf(M, ce_calls, fuse_qkv):
    l0, g0 = _train(M, False, fuse_qkv)
    assert ce_calls["n"] == 0
    l1, g1 = _train(M, True, fuse_qkv)
    assert ce_calls["n"] == 5
    assert max(abs(a - b) for a, b in zip(l0, l1)) <= 2e-2, (l0, l1)
    for a, b in zip(g0, g1):
        assert (a - b).abs().max().item() <= 0.05 * a.abs().max().item()


def _model(M, **kw):
    from transformers import LlamaForCausalLM
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg(**kw)).cuda().bfloat16()
    M.freeze_unselected_matrix_layer(model, {}, {("q_proj", 0): [(0, 1)]})
    M.convert_linear_layer_to_matrix_sparsity(model, {}, {("q_proj", 0): [(0, 1)]})
    return model


def test_fallbacks_take_the_hf_path(M, ce_calls):
    gen = torch.Generator().manual_seed(5)
    ids, labels = _batch(gen)

    model = _model(M)
    with torch.no_grad():
        ref = model(input_ids=ids, labels=labels, use_cache=False)
        assert M.fuse_causal_lm_loss(model)
        got = model(input_ids=ids, labels=labels, use_cache=False)
    assert ce_calls["n"] == 0 and torch.equal(got.logits, ref.logits) and torch.equal(got.loss, ref.loss)

    # logits_to_keep=1: HF's own path, logits of the last position only
    out = model(input_ids=ids, labels=labels[:, -1:], use_cache=False, logits_to_keep=1)
    assert ce_calls["n"] == 0 and out.logits.shape[1] == 1

    # return_dict=False on the native path: (loss,)
    tup = model(input_ids=ids, labels=labels, use_cache=False, return_dict=False)
    assert ce_calls["n"] == 1 and isinstance(tup, tuple) and tup[0].dim() == 0
    ref_loss = model(input_ids=ids, labels=labels, use_cache=False).loss
    assert ce_calls["n"] == 2 and torch.equal(tup[0], ref_loss)

    # a trainable lm_head: HF's path, and the lm_head gets its gradient
    model.lm_head.weight.requires_grad_(True)
    out = model(input_ids=ids, labels=labels, use_cache=False)
    out.loss.backward()
    assert ce_calls["n"] == 2 and out.logits is not None and model.lm_head.weight.grad is not None
    model.lm_head.weight.requires_grad_(False)

    # after unfuse_causal_lm_loss, the class's own forward
    assert M.unfuse_causal_lm_loss(model)
    out = model(input_ids=ids, labels=labels, use_cache=False)
    assert ce_calls["n"] == 2 and out.logits is not None
    assert torch.allclose(out.loss, ref_loss, rtol=2e-2)

    # a vocabulary the kernels do not take (32 001): HF's path, same result as the unfused model
    odd = _model(M, vocab_size=32001)
    ref = odd(input_ids=ids, labels=labels, use_cache=False)
    assert M.fuse_causal_lm_loss(odd)
    got = odd(input_ids=ids, labels=labels, use_cache=False)
    assert ce_calls["n"] == 2 and torch.equal(got.loss, ref.loss) and torch.equal(got.logits, ref.logits)


def test_num_items_in_batch_ignore_index_and_shift_labels(M, ce_calls):
    model = _model(M)
    gen = torch.Generator().manual_seed(6)
    ids, labels = _batch(gen)
    minus1 = labels.masked_fill(labels == -100, -1)
    shifted = torch.nn.functional.pad(minus1, (0, 1), value=-1)[:, 1:].contiguous()
    cases = [dict(labels=labels, num_items_in_batch=torch.tensor(100, device="cuda")),
             dict(labels=minus1, ignore_index=-1),
             dict(labels=minus1, shift_labels=shifted, ignore_index=-1)]
    for kw in cases:
        ref = model(input_ids=ids, use_cache=False, **kw).loss
        M.fuse_causal_lm_loss(model)
        n0 = ce_calls["n"]
        got = model(input_ids=ids, use_cache=False, **kw).loss
        assert ce_calls["n"] == n0 + 1, kw.keys()                    # the native path ran
        M.unfuse_causal_lm_loss(model)
        assert torch.allclose(got, ref, rtol=5e-3), (kw.keys(), got, ref)


def test_deepcopy_computes_with_the_copys_weights(M):
    model = _model(M)
    M.fuse_causal_lm_loss(model)
    twin = copy.deepcopy(model)
    gen = torch.Generator().manual_seed(7)
    ids, labels = _batch(gen)
    before = twin(input_ids=ids, labels=labels, use_cache=False).loss
    with torch.no_grad():
        model.lm_head.weight.mul_(-3.0)
    after = twin(input_ids=ids, labels=labels, use_cache=False).loss
    changed = model(input_ids=ids, labels=labels, use_cache=False).loss
    assert torch.equal(before, after) and not torch.equal(changed, before)
    assert twin.forward.__self__ is twin
