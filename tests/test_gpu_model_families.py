"""GPU tests of the Qwen3 / Mistral side of the fused decoder path: the per-head q/k RMSNorm + RoPE kernel
(`smt_qk_norm_rope_*`) against transformers' `Qwen3RMSNorm` + `apply_rotary_pos_emb`, SMT training of tiny Qwen3 and
Mistral models with and without the fused overrides, one Qwen3-8B-shaped layer against fp64, and the fused loss at a
vocabulary that is not a multiple of 256."""
import copy
import functools

import pytest
import torch

pytestmark = pytest.mark.gpu

HID, INTER, NQ, NKV, HD = 4096, 12288, 32, 8, 128           # Qwen3-8B widths
EPS = 1e-6


@pytest.fixture(scope="module")
def M(built_library):
    from sparse_matrix_tuning_b200.smt import smt
    return smt


def _tables(B, S, theta=1e6):
    pos = torch.arange(S, device="cuda").float()[:, None] * (theta ** (-torch.arange(0, HD, 2, device="cuda") / HD))
    emb = torch.cat((pos, pos), -1)[None]
    cos, sin = emb.cos().bfloat16(), emb.sin().bfloat16()
    return ((cos, sin), (cos.expand(B, -1, -1).contiguous(), sin.expand(B, -1, -1).contiguous()))


def _hf_norm(x, w, eps=EPS, rstd=None):
    """Qwen3RMSNorm's arithmetic; with `rstd` given, that value instead of its own."""
    xf = x.float()
    if rstd is None:
        rstd = torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)
    return w * (xf * rstd).to(x.dtype)


# ---- the kernel --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("heads", [(32, 8), (16, 8), (8, 8)])
def test_qk_norm_rope_forward_matches_hf(built_library, heads):
    from transformers.models.qwen3.modeling_qwen3 import Qwen3RMSNorm, apply_rotary_pos_emb
    from sparse_matrix_tuning_b200 import ops
    Hq, Hk = heads
    torch.manual_seed(0)
    B, S = 2, 512
    q = (torch.randn(B, S, Hq, HD, device="cuda") * 2).bfloat16()
    k = (torch.randn(B, S, Hk, HD, device="cuda") * 0.5).bfloat16()
    wq = (1 + 0.1 * torch.randn(HD, device="cuda")).bfloat16()
    wk = (1 + 0.1 * torch.randn(HD, device="cuda")).bfloat16()
    nq, nk = Qwen3RMSNorm(HD, EPS).cuda().bfloat16(), Qwen3RMSNorm(HD, EPS).cuda().bfloat16()
    with torch.no_grad():
        nq.weight.copy_(wq)
        nk.weight.copy_(wk)
        for cos, sin in _tables(B, S):
            q_ref, k_ref = apply_rotary_pos_emb(nq(q).transpose(1, 2), nk(k).transpose(1, 2), cos, sin)
            qo, ko, rq, rk = ops.qk_norm_rope_forward(q, k, wq, wk, EPS, EPS, cos, sin)
            for x, r in ((q, rq), (k, rk)):
                r_ref = torch.rsqrt(x.float().pow(2).mean(-1) + EPS).reshape(-1)
                assert torch.allclose(r, r_ref, rtol=1e-6, atol=0)
            # only the order of the row sum differs: HF's formula fed the kernel's rstd gives its output bit for bit
            q_own, k_own = apply_rotary_pos_emb(_hf_norm(q, wq, rstd=rq.view(B, S, Hq, 1)).transpose(1, 2),
                                                _hf_norm(k, wk, rstd=rk.view(B, S, Hk, 1)).transpose(1, 2), cos, sin)
            assert torch.equal(qo.transpose(1, 2), q_own) and torch.equal(ko.transpose(1, 2), k_own)
            for got, ref in ((qo.transpose(1, 2), q_ref), (ko.transpose(1, 2), k_ref)):
                assert (got == ref).float().mean().item() >= 0.999
            again = ops.qk_norm_rope_forward(q, k, wq, wk, EPS, EPS, cos, sin)
            assert all(torch.equal(a, b) for a, b in zip(again, (qo, ko, rq, rk)))


def test_qk_norm_rope_backward_no_worse_than_hf_against_fp64(built_library):
    from transformers.models.qwen3.modeling_qwen3 import apply_rotary_pos_emb
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(1)
    B, S = 2, 512
    q = (torch.randn(B, S, NQ, HD, device="cuda") * 2).bfloat16()
    k = torch.randn(B, S, NKV, HD, device="cuda").bfloat16()
    wq = (1 + 0.1 * torch.randn(HD, device="cuda")).bfloat16()
    wk = (1 + 0.1 * torch.randn(HD, device="cuda")).bfloat16()
    dq_o, dk_o = torch.randn_like(q), torch.randn_like(k)
    for cos, sin in _tables(B, S):
        q64, k64 = q.double().requires_grad_(True), k.double().requires_grad_(True)

        def norm64(x, w):
            return w.double() * x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + EPS)
        r64 = apply_rotary_pos_emb(norm64(q64, wq).transpose(1, 2), norm64(k64, wk).transpose(1, 2), cos.double(),
                                   sin.double())
        truth = torch.autograd.grad(r64, (q64, k64), (dq_o.double().transpose(1, 2), dk_o.double().transpose(1, 2)))
        qh, kh = q.clone().requires_grad_(True), k.clone().requires_grad_(True)
        rh = apply_rotary_pos_emb(_hf_norm(qh, wq).transpose(1, 2), _hf_norm(kh, wk).transpose(1, 2), cos, sin)
        hf = torch.autograd.grad(rh, (qh, kh), (dq_o.transpose(1, 2), dk_o.transpose(1, 2)))
        _qo, _ko, rq, rk = ops.qk_norm_rope_forward(q, k, wq, wk, EPS, EPS, cos, sin)
        got = ops.qk_norm_rope_backward(q, k, wq, wk, rq, rk, cos, sin, dq_o, dk_o)
        for t, h, g in zip(truth, hf, got):
            scale = t.abs().max().item()
            err, hf_err = [(x.double() - t).abs().max().item() / scale for x in (g, h)]
            assert err <= hf_err * 1.05 + 1e-6, (err, hf_err)


# ---- tiny models ---------------------------------------------------------------------------------------------------

def _cfg(family, **kw):
    import transformers
    base = dict(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
                num_key_value_heads=2, head_dim=128, max_position_embeddings=256, attn_implementation="sdpa")
    if family == "Mistral":
        base["sliding_window"] = 64                           # shorter than the sequences below
    base.update(kw)
    return getattr(transformers, f"{family}Config")(**base)


def _model(family, **kw):
    import transformers
    torch.manual_seed(0)
    return getattr(transformers, f"{family}ForCausalLM")(_cfg(family, **kw)).cuda().bfloat16()


def _train(M, family, fuse, sel_attn, sel_mlp, steps=3, lr=1e-3, padded=False, **kw):
    from sparse_matrix_tuning_b200.optim import SMTAdam
    model = _model(family, **kw)
    M.freeze_unselected_matrix_layer(model, sel_mlp, sel_attn)
    M.convert_linear_layer_to_matrix_sparsity(model, sel_mlp, sel_attn)
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    model.train()
    if fuse:
        assert M.fuse_qkv_projections(model) == 2 and M.fuse_causal_lm_loss(model)
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
            out = model(input_ids=ids, attention_mask=mask, position_ids=pos, labels=labels, use_cache=False)
            assert (out.logits is None) == fuse
            out.loss.backward()
            opt.step()
            losses.append(out.loss.item())
        params = torch.cat([opt.state[p]["master"].reshape(-1) for g in opt.param_groups for p in g["params"]])
        return losses, params
    finally:
        M.set_grouped_backward(False)
        M.unfuse_qkv_projections(model)
        M.unfuse_causal_lm_loss(model)


def _padded_batch(ids):
    """attention_mask, position_ids and labels for `ids` [2, S]: the first sequence left-padded by S // 4 tokens (HF's
    position ids cumsum(mask) - 1, padding at 1), the second three packed documents whose positions restart at 0."""
    B, S = ids.shape
    mask = torch.ones_like(ids)
    mask[0, :S // 4] = 0
    pos = (mask.cumsum(-1) - 1).masked_fill(mask == 0, 1)
    pos[1] = torch.cat([torch.arange(n, device=ids.device) for n in (S // 3, S // 3, S - 2 * (S // 3))])
    return mask, pos, ids.masked_fill(mask == 0, -100)


_TRAIN_CASES = [("Qwen3", False, False, False), ("Qwen3", True, False, False), ("Qwen3", True, True, False),
                ("Mistral", False, False, False), ("Mistral", True, False, False), ("Qwen3", True, False, True),
                ("Mistral", True, False, True)]


@pytest.mark.parametrize("family,with_mlp,tied,padded", _TRAIN_CASES,
                         ids=["-".join(map(str, c[:3])) + ("-padded" if c[3] else "") for c in _TRAIN_CASES])
def test_tiny_smt_training_fused_matches_unfused(M, family, with_mlp, tied, padded):
    sel_attn = {("q_proj", 0): [(0, 1), (1, 0)], ("k_proj", 0): [(0, 0)], ("v_proj", 1): [(0, 1)],
                ("q_proj", 1): [(1, 1)]}
    sel_mlp = {("gate_proj", 0): [(1, 0), (3, 1)], ("up_proj", 1): [(2, 0)], ("down_proj", 0): [(0, 2)]} \
        if with_mlp else {}
    steps, lr = 3, 1e-3
    l0, p0 = _train(M, family, False, sel_attn, sel_mlp, steps, lr, padded, tie_word_embeddings=tied)
    l1, p1 = _train(M, family, True, sel_attn, sel_mlp, steps, lr, padded, tie_word_embeddings=tied)
    assert max(abs(a - b) for a, b in zip(l0, l1)) <= 1e-2, (l0, l1)
    assert (p1 - p0).abs().max().item() <= 2 * steps * lr


@pytest.mark.parametrize("family", ["Llama", "Mistral", "Qwen3"])
def test_attention_override_passes_the_family_sliding_window(M, monkeypatch, family):
    """SDPA takes the window from the mask, so only a spy on the interface sees a dropped `sliding_window`."""
    from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS
    seen = []
    sdpa = ALL_ATTENTION_FUNCTIONS["sdpa"]

    def spy(module, *a, **k):
        seen.append(k.get("sliding_window", "absent"))
        return sdpa(module, *a, **k)
    monkeypatch.setitem(ALL_ATTENTION_FUNCTIONS._local_mapping, "sdpa", spy)
    kw = dict(use_sliding_window=True, sliding_window=32, max_window_layers=1) if family == "Qwen3" else {}
    model = _model(family, **kw)
    M.freeze_unselected_matrix_layer(model, {}, {})
    ids = torch.randint(0, 512, (2, 96), generator=torch.Generator().manual_seed(2)).cuda()
    with torch.no_grad():
        ref = model(input_ids=ids, use_cache=False).logits
        hf_seen, seen[:] = list(seen), []
        assert M.fuse_qkv_projections(model) == 2 and "forward" in model.model.layers[0].self_attn.__dict__
        fused = model(input_ids=ids, use_cache=False).logits
    assert seen == hf_seen
    assert hf_seen == {"Llama": ["absent"] * 2, "Mistral": [64] * 2, "Qwen3": [None, 32]}[family]
    assert (fused.float() - ref.float()).abs().max().item() <= 0.05 * ref.float().abs().max().item()


def test_fused_qwen3_step_never_calls_hf_norm_or_rope(M, monkeypatch):
    from transformers.models.qwen3 import modeling_qwen3 as Q
    model = _model("Qwen3")
    sel = {("q_proj", 0): [(0, 1)], ("k_proj", 1): [(0, 0)]}
    M.freeze_unselected_matrix_layer(model, {}, sel)
    M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    assert M.fuse_qkv_projections(model) == 2 and M.fuse_causal_lm_loss(model)
    calls = {"norm": 0, "rope": 0}
    norm_fwd, rope = Q.Qwen3RMSNorm.forward, Q.apply_rotary_pos_emb

    @functools.wraps(norm_fwd)
    def norm_spy(*a, **k):
        calls["norm"] += 1
        return norm_fwd(*a, **k)

    @functools.wraps(rope)
    def rope_spy(*a, **k):
        calls["rope"] += 1
        return rope(*a, **k)
    monkeypatch.setattr(Q.Qwen3RMSNorm, "forward", norm_spy)
    monkeypatch.setattr(Q, "apply_rotary_pos_emb", rope_spy)
    ids = torch.randint(0, 512, (2, 128), generator=torch.Generator().manual_seed(3)).cuda()
    out = model(input_ids=ids, labels=ids, use_cache=False)
    out.loss.backward()
    assert calls == {"norm": 0, "rope": 0} and torch.isfinite(out.loss)
    # the same spies do see the unfused model's calls
    M.unfuse_qkv_projections(model)
    model(input_ids=ids, labels=ids, use_cache=False)
    assert calls["norm"] > 0 and calls["rope"] > 0


def test_decoder_layer_at_qwen3_8b_widths_against_fp64(M):
    """One Qwen3-8B-shaped layer with SMT q/k/v blocks under non-reentrant checkpointing: output, dx and the compact
    block gradients of the fused layer are no further from an fp64 truth than the HF layer's."""
    from torch.utils.checkpoint import checkpoint
    from transformers.models.qwen3.modeling_qwen3 import Qwen3DecoderLayer, Qwen3RotaryEmbedding
    cfg = _cfg("Qwen3", hidden_size=HID, intermediate_size=INTER, num_attention_heads=NQ, num_key_value_heads=NKV,
               num_hidden_layers=1, max_position_embeddings=512, rms_norm_eps=EPS, rope_theta=1e6)
    torch.manual_seed(5)
    base = Qwen3DecoderLayer(cfg, 0).cuda()
    with torch.no_grad():
        for n, p in base.named_parameters():
            p.copy_(1 + 0.1 * torch.randn_like(p) if "norm" in n else torch.randn_like(p) * 0.02)
    B, S = 2, 256
    x = torch.randn(B, S, HID, device="cuda")
    dout = torch.randn(B, S, HID, device="cuda")
    rope = Qwen3RotaryEmbedding(cfg).cuda()
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


# ---- the fused loss at a vocabulary off the 256 grid ---------------------------------------------------------------

@pytest.fixture
def mm_calls(monkeypatch):
    """Counts library GEMMs issued through `torch.mm` (the vocabulary tail of `LinearCrossEntropyFn`)."""
    calls = {"n": 0}
    mm = torch.mm

    def wrapped(*a, **k):
        calls["n"] += 1
        return mm(*a, **k)
    monkeypatch.setattr(torch, "mm", wrapped)
    return calls


@pytest.mark.parametrize("family,V", [("Qwen3", 1216), ("Qwen3", 1024), ("Llama", 32064)],
                         ids=["1216", "1024", "Llama-32064"])
def test_fused_loss_at_a_vocabulary_off_the_256_grid(M, mm_calls, family, V):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    model = _model(family, vocab_size=V, num_hidden_layers=1)
    for p in model.parameters():
        p.requires_grad_(False)
    model.enable_input_require_grads()
    ids = torch.randint(0, V, (4, 1536), generator=torch.Generator().manual_seed(4)).cuda()
    labels = ids.clone()
    labels[:, ::5] = -100
    h = model.model(input_ids=ids).last_hidden_state.detach()

    def hf():
        x = h.clone().requires_grad_(True)
        loss = model.loss_function(logits=model.lm_head(x), labels=labels, vocab_size=V)
        loss.backward()
        return loss.detach(), x.grad

    ref_loss, ref_dh = hf()
    n0 = mm_calls["n"]
    x = h.clone().requires_grad_(True)
    loss = D.causal_lm_loss(x, model.lm_head.weight, labels)
    loss.backward()
    chunks = -(-ids.numel() // D._CE_CHUNK_ROWS)
    assert mm_calls["n"] - n0 == (chunks if V % 256 else 0)
    assert torch.allclose(loss, ref_loss, rtol=5e-3), (loss.item(), ref_loss.item())
    scale = ref_dh.float().abs().max().item()
    assert (x.grad.float() - ref_dh.float()).abs().max().item() <= 0.05 * scale
    # through the model override: logits=None and the same loss
    assert M.fuse_causal_lm_loss(model)
    out = model(input_ids=ids, labels=labels, use_cache=False)
    assert out.logits is None and torch.allclose(out.loss, ref_loss, rtol=5e-3)


def _ce_fp64(h, w, y):
    """Mean causal-LM cross-entropy over the labels that are not -100 and its input gradient, in fp64."""
    logits = h.double() @ w.double().T
    valid = y != -100
    denom = valid.sum().double()
    rows = (torch.logsumexp(logits, -1) - logits.gather(1, y.clamp_min(0)[:, None])[:, 0]) * valid
    p = torch.softmax(logits, -1)
    p[torch.arange(len(y), device="cuda"), y.clamp_min(0)] -= 1
    return rows.sum() / denom, ((p * valid[:, None]) / denom) @ w.double()


def _ce_pair(h, w, y, fn):
    hg = h.clone().requires_grad_(True)
    loss = fn(hg)
    loss.backward()
    return loss.detach(), hg.grad


@pytest.mark.parametrize("V,K", [(1216, 512), (151936, 4096)])
def test_linear_cross_entropy_off_the_256_grid_against_fp64(built_library, V, K):
    """The vocabulary tail (the last V % 256 columns, one library GEMM per chunk) held to the criterion of
    `test_linear_cross_entropy_no_worse_than_hf_against_fp64`: loss and dh against fp64, no worse than 1.5x HF's error
    (+ 1e-4 of the loss).  Once over all labels (a third of them in the tail), once over tail labels only, where a tail
    computed from the wrong weight rows, left at zero or never written fails by a wide margin."""
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    T = 2560                                                  # two chunks, the last one ragged
    g = torch.Generator(device="cuda").manual_seed(9)
    h = torch.randn(T, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(V, K, device="cuda", generator=g) * (1.5 / K ** 0.5)).bfloat16()
    V0 = V - V % 256
    y = torch.randint(0, V0, (T,), device="cuda", generator=g)
    tail = torch.arange(T, device="cuda") % 3 == 0
    y[tail] = torch.randint(V0, V, (int(tail.sum()),), device="cuda", generator=g)
    y[torch.rand(T, device="cuda", generator=g) < 0.2] = -100
    for labels in (y, torch.where(tail, y, torch.full_like(y, -100))):
        loss64, dh64 = _ce_fp64(h, w, labels)
        hf_loss, hf_dh = _ce_pair(h, w, labels, lambda x: torch.nn.functional.cross_entropy(
            torch.nn.functional.linear(x, w).float(), labels, ignore_index=-100))
        loss, dh = _ce_pair(h, w, labels, lambda x: D.LinearCrossEntropyFn.apply(
            x, w, labels, (labels != -100).sum(), -100))
        e_hf, e = (hf_loss.double() - loss64).abs().item(), (loss.double() - loss64).abs().item()
        assert e <= 1.5 * e_hf + 1e-4 * loss64.abs().item(), (e, e_hf, loss64.item())
        d_hf, d = (hf_dh.double() - dh64).abs().max().item(), (dh.double() - dh64).abs().max().item()
        assert d <= 1.5 * d_hf, (d, d_hf)


# ---- fallbacks and lifecycle ---------------------------------------------------------------------------------------

def test_kv_cache_and_trainable_qk_norm_run_hf_code(M):
    from transformers import DynamicCache
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    model = _model("Qwen3")
    M.freeze_unselected_matrix_layer(model, {}, {})
    M.fuse_qkv_projections(model)
    model.eval()
    layer = model.model.layers[0]
    h = torch.randn(2, 16, 512, device="cuda").bfloat16()
    pos = torch.arange(16, device="cuda")[None]
    pe = model.model.rotary_emb(h, pos)
    with torch.no_grad():
        got = layer(h, position_embeddings=pe, position_ids=pos, past_key_values=DynamicCache(config=model.config),
                    use_cache=True)
        D.remove_all(model)
        ref = layer(h, position_embeddings=pe, position_ids=pos, past_key_values=DynamicCache(config=model.config),
                    use_cache=True)
    assert torch.equal(got, ref)

    # a trainable q_norm: the attention runs the class's own forward and the norm weight gets its gradient
    attn = layer.self_attn
    attn.q_norm.weight.requires_grad_(True)
    hq = h.clone().requires_grad_(True)
    ref = attn(hq, position_embeddings=pe, attention_mask=None)[0]
    ref.float().sum().backward()
    g_ref = attn.q_norm.weight.grad.clone()
    attn.q_norm.weight.grad = None
    assert D.install_layer(layer)
    got = attn(hq, position_embeddings=pe, attention_mask=None)[0]
    got.float().sum().backward()
    assert torch.equal(got, ref) and torch.equal(attn.q_norm.weight.grad, g_ref)
    M.unfuse_qkv_projections(model)


def test_unfuse_and_deepcopy_of_a_fused_qwen3_model(M):
    model = _model("Qwen3")
    sel = {("q_proj", 0): [(0, 1)], ("k_proj", 1): [(0, 0)]}
    M.freeze_unselected_matrix_layer(model, {}, sel)
    M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    ids = torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(6)).cuda()
    with torch.no_grad():
        ref = model(input_ids=ids, use_cache=False).logits
        assert M.fuse_qkv_projections(model) == 2
        fused = model(input_ids=ids, use_cache=False).logits
        twin = copy.deepcopy(model)
        saved = {n: p.detach().clone() for n, p in model.named_parameters()}
        before = twin(input_ids=ids, use_cache=False).logits
        assert torch.equal(before, fused)
        for n, p in model.named_parameters():                    # q/k/v (dense and compact) and every norm
            if any(k in n for k in ("q_proj", "k_proj", "v_proj", "norm")):
                p.mul_(-3.0)
        after = twin(input_ids=ids, use_cache=False).logits
        changed = model(input_ids=ids, use_cache=False).logits
        assert torch.equal(before, after) and not torch.equal(changed, before)
        for n, p in model.named_parameters():
            p.copy_(saved[n])
        assert M.unfuse_qkv_projections(model) == 2
        assert not [n for n, m in model.named_modules() if "forward" in m.__dict__]
        again = model(input_ids=ids, use_cache=False).logits
    assert torch.equal(again, ref)
    assert (fused.float() - ref.float()).abs().max().item() <= 0.05 * ref.float().abs().max().item()
