"""GPU tests of the decoder-layer elementwise kernels (csrc/decoder_kernels.cu) and of their installation on a
transformers LLaMA model by `fuse_qkv_projections` (decoder_fusion.py)."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu

HID, INTER, NQ, NKV, HD = 4096, 14336, 32, 8, 128          # LLaMA-3-8B widths


@pytest.fixture(scope="module")
def M(built_library):
    from sparse_matrix_tuning_b200.smt import smt
    return smt


@pytest.fixture
def spy(monkeypatch, built_library):
    """Counts calls of the forward entry points of the decoder kernels."""
    from sparse_matrix_tuning_b200 import ops
    calls = {"rmsnorm_forward": 0, "rope_forward": 0, "swiglu_forward": 0}
    for name in calls:
        fn = getattr(ops, name)

        def wrapped(*a, _fn=fn, _name=name, **k):
            calls[_name] += 1
            return _fn(*a, **k)
        monkeypatch.setattr(ops, name, wrapped)
    return calls


def _ulp_bf16(x):
    """Spacing of bf16 numbers at |x| (fp32 tensor)."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def _hf_rmsnorm(x, w, eps):
    xf = x.float()
    return w * (xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)).to(x.dtype)


# ---- per kernel, LLaMA-3-8B widths --------------------------------------------------------------------------------

def test_rope_forward_and_backward_bit_exact_vs_hf(built_library):
    from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(0)
    B, S = 2, 512
    q = torch.randn(B, S, NQ, HD, device="cuda").bfloat16()
    k = torch.randn(B, S, NKV, HD, device="cuda").bfloat16()
    pos = torch.arange(S, device="cuda").float()[:, None] * (500000.0 ** (-torch.arange(0, HD, 2, device="cuda") / HD))
    emb = torch.cat((pos, pos), -1)[None]
    cos, sin = emb.cos().bfloat16(), emb.sin().bfloat16()
    for cs in ((cos, sin), (cos.expand(B, -1, -1).contiguous(), sin.expand(B, -1, -1).contiguous())):
        qt, kt = q.transpose(1, 2).requires_grad_(True), k.transpose(1, 2).requires_grad_(True)
        q_ref, k_ref = apply_rotary_pos_emb(qt, kt, *cs)
        q_got, k_got = ops.rope_forward(q, k, *cs)
        assert torch.equal(q_got.transpose(1, 2), q_ref) and torch.equal(k_got.transpose(1, 2), k_ref)
        dq_out, dk_out = torch.randn_like(q), torch.randn_like(k)
        dq_ref, dk_ref = torch.autograd.grad((q_ref, k_ref), (qt, kt), (dq_out.transpose(1, 2), dk_out.transpose(1, 2)))
        dq, dk = ops.rope_backward(dq_out, dk_out, *cs)
        assert torch.equal(dq.transpose(1, 2), dq_ref) and torch.equal(dk.transpose(1, 2), dk_ref)


def test_swiglu_forward_bit_exact_backward_within_one_ulp(built_library):
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(1)
    g = (torch.randn(1024, INTER, device="cuda") * 3).bfloat16().requires_grad_(True)
    u = torch.randn(1024, INTER, device="cuda").bfloat16().requires_grad_(True)
    h_ref = torch.nn.functional.silu(g) * u
    assert torch.equal(ops.swiglu_forward(g.detach(), u.detach()), h_ref)
    dh = torch.randn_like(h_ref)
    dg_ref, du_ref = torch.autograd.grad(h_ref, (g, u), dh)
    dg, du = ops.swiglu_backward(g.detach(), u.detach(), dh)
    for got, ref in ((dg, dg_ref), (du, du_ref)):
        diff = (got.float() - ref.float()).abs()
        assert (diff <= _ulp_bf16(ref.float())).all(), diff.max().item()


@pytest.mark.parametrize("residual", [False, True])
def test_rmsnorm_forward_matches_hf(built_library, residual):
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(2)
    T, eps = 4096, 1e-5
    a = torch.randn(T, HID, device="cuda").bfloat16()
    res = torch.randn(T, HID, device="cuda").bfloat16() if residual else None
    w = (1 + 0.1 * torch.randn(HID, device="cuda")).bfloat16()
    x = (res + a) if residual else a
    y_ref = _hf_rmsnorm(x, w, eps)
    y, rstd, h = ops.rmsnorm_forward(a, w, eps, res=res)
    if residual:
        assert torch.equal(h, x)
    assert (y == y_ref).float().mean().item() >= 0.999
    # only the order of the row sum differs: with the kernel's own rstd, HF's formula gives the kernel's output bit for
    # bit, and the bf16 normalised value it rounds through is within one bf16 ulp of HF's
    rstd_ref = torch.rsqrt(x.float().pow(2).mean(-1) + eps)
    assert torch.allclose(rstd, rstd_ref, rtol=1e-6, atol=0)
    n_ref, n_got = (x.float() * rstd_ref[:, None]).bfloat16(), (x.float() * rstd[:, None]).bfloat16()
    assert torch.equal(y, w * n_got)
    assert ((n_got.float() - n_ref.float()).abs() <= _ulp_bf16(n_ref.float())).all()
    y2, rstd2, _ = ops.rmsnorm_forward(a, w, eps, res=res)
    assert torch.equal(y, y2) and torch.equal(rstd, rstd2)                 # deterministic (recomputation)


@pytest.mark.parametrize("with_dres", [False, True])
def test_rmsnorm_backward_no_worse_than_hf_against_fp64(built_library, with_dres):
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(3)
    T, eps = 2048, 1e-5
    x = torch.randn(T, HID, device="cuda").bfloat16()
    w = (1 + 0.1 * torch.randn(HID, device="cuda")).bfloat16()
    dy = torch.randn(T, HID, device="cuda").bfloat16()
    dres = torch.randn(T, HID, device="cuda").bfloat16() if with_dres else None
    x64 = x.double().requires_grad_(True)
    y64 = w.double() * (x64 * torch.rsqrt(x64.pow(2).mean(-1, keepdim=True) + eps))
    truth = torch.autograd.grad(y64, x64, dy.double())[0] + (dres.double() if with_dres else 0)
    xh = x.clone().requires_grad_(True)
    hf = torch.autograd.grad(_hf_rmsnorm(xh, w, eps), xh, dy)[0]
    if with_dres:
        hf = hf + dres                                                       # autograd's bf16 add at the fork
    _y, rstd, _ = ops.rmsnorm_forward(x, w, eps)
    got = ops.rmsnorm_backward(x, w, rstd, dy, dres)
    scale = truth.abs().max().item()
    err, hf_err = [(t.double() - truth).abs().max().item() / scale for t in (got, hf)]
    assert err <= hf_err * 1.05 + 1e-6, (err, hf_err)


# ---- models --------------------------------------------------------------------------------------------------------

def _tiny_cfg(**kw):
    from transformers import LlamaConfig
    base = dict(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
                num_key_value_heads=2, head_dim=128, max_position_embeddings=256, attn_implementation="sdpa")
    base.update(kw)
    return LlamaConfig(**base)


def _train(M, fuse, sel_attn, sel_mlp, steps=3, lr=1e-3, padded=False):
    from transformers import LlamaForCausalLM
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda().bfloat16()
    M.freeze_unselected_matrix_layer(model, sel_mlp, sel_attn)
    M.convert_linear_layer_to_matrix_sparsity(model, sel_mlp, sel_attn)
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    model.train()
    if fuse:
        assert M.fuse_qkv_projections(model) == 2
        assert "forward" in model.model.layers[0].__dict__ and "forward" in model.model.norm.__dict__
    opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, lr), betas=(0.9, 0.95), max_grad_norm=1.0)
    M.set_grouped_backward(True)
    try:
        gen = torch.Generator().manual_seed(1)
        losses = []
        for _ in range(steps):
            ids = torch.randint(0, 512, (2, 128), generator=gen).cuda()
            mask, pos, labels = _padded_batch(ids) if padded else (None, None, ids)
            opt.zero_grad()
            loss = model(input_ids=ids, attention_mask=mask, position_ids=pos, labels=labels, use_cache=False).loss
            loss.backward()
            opt.step()
            losses.append(loss.item())
        params = torch.cat([opt.state[p]["master"].reshape(-1) for g in opt.param_groups for p in g["params"]])
        return losses, params
    finally:
        M.set_grouped_backward(False)
        M.unfuse_qkv_projections(model)


def _padded_batch(ids):
    """attention_mask, position_ids and labels for `ids` [2, S]: the first sequence left-padded by S // 4 tokens (HF's
    position ids cumsum(mask) - 1, padding at 1), the second three packed documents whose positions restart at 0."""
    B, S = ids.shape
    mask = torch.ones_like(ids)
    mask[0, :S // 4] = 0
    pos = (mask.cumsum(-1) - 1).masked_fill(mask == 0, 1)
    pos[1] = torch.cat([torch.arange(n, device=ids.device) for n in (S // 3, S // 3, S - 2 * (S // 3))])
    return mask, pos, ids.masked_fill(mask == 0, -100)


@pytest.mark.parametrize("with_mlp,padded", [(False, False), (True, False), (True, True)],
                         ids=["False", "True", "True-padded"])
def test_tiny_llama_smt_training_fused_matches_unfused(M, with_mlp, padded):
    sel_attn = {("q_proj", 0): [(0, 1), (1, 0)], ("k_proj", 0): [(0, 0)], ("v_proj", 1): [(0, 1)],
                ("q_proj", 1): [(1, 1)]}
    sel_mlp = {("gate_proj", 0): [(1, 0), (3, 1)], ("up_proj", 1): [(2, 0)], ("down_proj", 0): [(0, 2)]} \
        if with_mlp else {}
    steps, lr = 3, 1e-3
    l0, p0 = _train(M, False, sel_attn, sel_mlp, steps, lr, padded)
    l1, p1 = _train(M, True, sel_attn, sel_mlp, steps, lr, padded)
    assert max(abs(a - b) for a, b in zip(l0, l1)) <= 1e-2, (l0, l1)
    assert (p1 - p0).abs().max().item() <= 2 * steps * lr


def test_decoder_layer_at_llama3_8b_widths_against_fp64(M):
    """One LLaMA-3-8B-shaped layer with SMT q/k/v blocks under non-reentrant checkpointing: output, dx and the compact
    block gradients of the fused layer are no further from an fp64 truth than the HF layer's."""
    from torch.utils.checkpoint import checkpoint
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer, LlamaRotaryEmbedding
    cfg = _tiny_cfg(hidden_size=HID, intermediate_size=INTER, num_attention_heads=NQ, num_key_value_heads=NKV,
                    num_hidden_layers=1, max_position_embeddings=512)
    torch.manual_seed(5)
    base = LlamaDecoderLayer(cfg, 0).cuda()
    with torch.no_grad():
        for n, p in base.named_parameters():
            p.copy_(1 + 0.1 * torch.randn_like(p) if "norm" in n else torch.randn_like(p) * 0.02)
    B, S = 2, 256
    x = torch.randn(B, S, HID, device="cuda")
    dout = torch.randn(B, S, HID, device="cuda")
    rope = LlamaRotaryEmbedding(cfg).cuda()
    pos = torch.arange(S, device="cuda")[None]
    sel = {"q_proj": [(0, 1), (5, 3), (15, 15)], "k_proj": [(1, 2), (3, 0)], "v_proj": [(2, 7)]}

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
        out = checkpoint(lambda t: layer(t, position_embeddings=pe, position_ids=pos), xin, use_reentrant=False)
        out.backward(dout.to(dtype))
        if dtype == torch.float64:
            blocks = [getattr(attn, n).weight.grad[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256]
                      for n, idx in sel.items() for r, c in idx]
        else:
            blocks = [getattr(attn, n).selected_weight.grad.view(-1, 256, 256)[i]
                      for n, idx in sel.items() for i in range(len(idx))]
        return out.detach().double(), xin.grad.double(), torch.stack(blocks).double()

    truth = run(torch.float64, False)
    hf = run(torch.bfloat16, False)
    fused = run(torch.bfloat16, True)
    for what, t, h, f in zip(("output", "dx", "block grads"), truth, hf, fused):
        scale = t.abs().max().item()
        e_hf, e_f = (h - t).abs().max().item() / scale, (f - t).abs().max().item() / scale
        assert e_f <= e_hf * 1.25 + 1e-4, (what, e_f, e_hf)


def _fwd_bwd(model, ids):
    from sparse_matrix_tuning_b200 import ops
    n0 = ops.LAUNCHES["total"]
    out = model(input_ids=ids, labels=ids, use_cache=False)
    out.loss.backward()
    return out.logits.detach(), ops.LAUNCHES["total"] - n0


def test_fallbacks_take_the_hf_path(M, spy):
    from transformers import DynamicCache, LlamaForCausalLM
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    ids = torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(2)).cuda()

    # fp32 model with the overrides installed by hand: every piece falls back, bit-identical to HF, no launch
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda()
    ref, _ = _fwd_bwd(model, ids)
    assert all(D.install_layer(l) for l in model.model.layers) and D.install_norm(model.model.norm)
    got, launches = _fwd_bwd(model, ids)
    assert torch.equal(got, ref) and launches == 0 and sum(spy.values()) == 0
    D.remove_all(model)

    # head_dim != 128: fuse_qkv_projections fuses the projections but leaves the layer's elementwise ops to HF
    model = LlamaForCausalLM(_tiny_cfg(head_dim=64, num_attention_heads=8, num_key_value_heads=4)).cuda().bfloat16()
    M.freeze_unselected_matrix_layer(model, {}, {})
    with pytest.warns(UserWarning):
        assert M.fuse_qkv_projections(model) == 2
    assert "forward" not in model.model.layers[0].__dict__ and "forward" not in model.model.norm.__dict__
    with torch.no_grad():
        model(input_ids=ids, use_cache=False)
    assert sum(spy.values()) == 0
    M.unfuse_qkv_projections(model)

    # trainable norm weights: the norms run HF's code (their weights get gradients), RoPE and SwiGLU stay native
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda().bfloat16()
    M.freeze_unselected_matrix_layer(model, {}, {})
    for n, p in model.named_parameters():
        p.requires_grad_("norm" in n)
    M.fuse_qkv_projections(model)
    _fwd_bwd(model, ids)
    assert spy["rmsnorm_forward"] == 0 and spy["rope_forward"] > 0 and spy["swiglu_forward"] > 0
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for n, p in model.named_parameters() if "norm" in n)

    # a KV cache: the whole layer (norms and MLP included) runs HF's code, bit-identical to the layer without the
    # elementwise overrides (the q/k/v projections stay fused in both)
    for p in model.parameters():
        p.requires_grad_(False)
    model.eval()
    for k in spy:
        spy[k] = 0
    layer = model.model.layers[0]
    h = torch.randn(2, 16, 512, device="cuda").bfloat16()
    pos = torch.arange(16, device="cuda")[None]
    pe = model.model.rotary_emb(h, pos)
    with torch.no_grad():
        got = layer(h, position_embeddings=pe, position_ids=pos, past_key_values=DynamicCache(config=model.config),
                    use_cache=True)
        assert D.remove_all(model) == 2
        ref = layer(h, position_embeddings=pe, position_ids=pos, past_key_values=DynamicCache(config=model.config),
                    use_cache=True)
    assert sum(spy.values()) == 0 and torch.equal(got, ref)


def test_unfuse_restores_bit_identical_hf_outputs(M, spy):
    from transformers import LlamaForCausalLM
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda().bfloat16()
    M.freeze_unselected_matrix_layer(model, {}, {})
    ids = torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(3)).cuda()
    with torch.no_grad():
        ref = model(input_ids=ids, use_cache=False).logits
        assert M.fuse_qkv_projections(model) == 2
        fused = model(input_ids=ids, use_cache=False).logits
        assert spy["rope_forward"] == 2 and spy["swiglu_forward"] == 2 and spy["rmsnorm_forward"] == 5
        assert M.unfuse_qkv_projections(model) == 2
        assert not [n for n, m in model.named_modules() if "forward" in m.__dict__]
        again = model(input_ids=ids, use_cache=False).logits
    assert torch.equal(again, ref)
    assert (fused.float() - ref.float()).abs().max().item() <= 0.05 * ref.float().abs().max().item()


def test_deepcopy_of_a_fused_model_computes_with_the_copys_weights(M):
    from transformers import LlamaForCausalLM
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda().bfloat16()
    sel = {("q_proj", 0): [(0, 1)], ("k_proj", 1): [(0, 0)]}
    M.freeze_unselected_matrix_layer(model, {}, sel)
    M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    M.fuse_qkv_projections(model)
    twin = copy.deepcopy(model)
    ids = torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(4)).cuda()
    with torch.no_grad():
        before = twin(input_ids=ids, use_cache=False).logits
        for n, p in model.named_parameters():                    # q/k/v (dense and compact) and the norms
            if any(k in n for k in ("q_proj", "k_proj", "v_proj", "norm")):
                p.mul_(-3.0)
        after = twin(input_ids=ids, use_cache=False).logits
        changed = model(input_ids=ids, use_cache=False).logits
    assert torch.equal(before, after)
    assert not torch.equal(changed, before)
    layer = twin.model.layers[1]
    assert layer.forward.__self__ is layer and layer.self_attn.q_proj.forward.__self__ is layer.self_attn.q_proj
    assert layer.self_attn.q_proj._smt_shared_group.members[0] is layer.self_attn.q_proj
