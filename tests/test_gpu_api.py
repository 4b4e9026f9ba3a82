"""GPU parity tests, API level: the drop-in `smt` package (same names as the reference's deepspeed/smt/*.py) is fed
the inputs the committed golden vectors were generated from — by the UNMODIFIED reference, see
oracle/gen_golden.py — and must reproduce the reference's outputs: selected indices exactly (dict order and list
order included), tensors within the stated tolerances."""
import pytest
import torch

from conftest import load_golden
from oracle import golden_inputs as GI
from oracle import smt_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api(built_library):
    from sparse_matrix_tuning_b200.smt import smt as M, smt_helper as H
    return M, H


@pytest.mark.parametrize("case", load_golden("selection_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_select_submatrix_golden(api, case):
    _M, H = api
    spec = case["spec"]
    grads, dims = GI.make_selection_inputs(spec)
    assert GI.tensor_dict_sha(grads) == case["input_sha"]
    kw = dict(selection_strategy=spec["selection_strategy"], calculate_strategy=spec["calculate_strategy"])
    if "raises" in case:                                           # n == 0: the reference dies with UnboundLocalError
        with pytest.raises(UnboundLocalError):
            H.select_submatrix_based_on_grads(grads, dims, spec["n"], **kw)
        return
    # host buffers in (the reference's capture loop leaves the sums on the CPU), indices out
    got = H.select_submatrix_based_on_grads(grads, dims, spec["n"], **kw)
    assert isinstance(got, dict) and got.default_factory is list
    assert [(k, list(v)) for k, v in got.items()] == [(k, [tuple(t) for t in v]) for k, v in case["selection"]]
    # same call with device-resident accumulators
    got_dev = H.select_submatrix_based_on_grads({k: g.cuda() for k, g in grads.items()}, dims, spec["n"], **kw)
    assert list(got_dev.items()) == list(got.items())


@pytest.mark.parametrize("case", load_golden("channel_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_select_channels_golden(api, case):
    _M, H = api
    spec = case["spec"]
    act = GI.make_channel_inputs(spec)
    assert GI.tensor_dict_sha(act) == case["input_sha"]
    got = H.select_channel_based_on_activation(act, n=spec["n"], selection_strategy=spec["selection_strategy"],
                                               calculate_strategy=spec["calculate_strategy"])
    want = {k: list(v) for k, v in case["selection"]}
    if spec["selection_strategy"] == "norm_dist" or spec["name"] == "planted":
        # planted/norm_dist cases contain exact score ties inside one matrix where the reference's order comes from
        # Python tuple order (heap) or an unstable argsort: compare as sets per key plus the tie-free prefix order
        assert {k: sorted(v) for k, v in got.items()} == {k: sorted(v) for k, v in want.items()}
    else:
        assert [(k, list(v)) for k, v in got.items()] == [(k, v) for k, v in want.items()]


def test_select_channels_planted_order_is_tuple_order(api):
    """The planted example of smt_helper.py:323-338: ties are resolved by Python tuple order, larger tuple first."""
    _M, H = api
    case = [c for c in load_golden("channel_cases.pt") if c["spec"]["name"] == "planted"][0]
    act = GI.make_channel_inputs(case["spec"])
    got = H.select_channel_based_on_activation(act, n=case["spec"]["n"])
    assert [(k, list(v)) for k, v in got.items()] == [(k, list(v)) for k, v in case["selection"]]


@pytest.mark.parametrize("case", load_golden("linearz_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_linear_layer_matrix_sparsity_golden(api, case):
    M, _H = api
    spec, b = case["spec"], case["spec"]["block"]
    x, dy, w, idx = case["x"], case["dy"], case["w"], case["index_list"]
    M.Block_dimension = b
    try:
        layer = M.LinearLayer_MatrixSparsity(torch.nn.Parameter(w.clone().cuda()), bias=None, index_list=idx)
        assert torch.equal(layer.selected_weight.detach().cpu(), case["selected0"])          # gather: exact
        assert layer.selected_weight.requires_grad and not layer.weight.requires_grad
        with torch.no_grad():
            layer.selected_weight.mul_(0.5)                                                  # as in gen_golden.py
        xin = x.clone().cuda().requires_grad_(True)
        y = layer(xin)
        assert GI.tensor_dict_sha({"w": layer.weight.detach().cpu()}) == case["w_after_sha"]  # scatter: exact
        y.backward(dy.cuda())
    finally:
        M.Block_dimension = 256
    gw, gi = layer.selected_weight.grad.cpu(), xin.grad.cpu()
    assert gw.shape == case["grad_weight"].shape and gw.dtype == case["grad_weight"].dtype
    w2 = O.scatter_blocks(w.clone(), case["selected0"] * 0.5, idx, b)
    truth = O.block_grad_truth(x, dy, idx, b)
    scale = truth.abs().max().item()
    if spec["dtype"] == "float32":
        assert (gw - case["grad_weight"]).abs().max().item() <= 1e-5 * scale
        assert torch.allclose(y.detach().cpu(), case["y"], rtol=1e-4, atol=1e-5)             # dense side: cuBLAS vs CPU
        assert torch.allclose(gi, case["grad_input"], rtol=1e-4, atol=1e-5)
    else:
        err = (gw.double() - truth).abs().max().item() / scale
        ref_err = (case["grad_weight"].double() - truth).abs().max().item() / scale
        assert err <= 2 ** -7 and err <= ref_err * 1.10 + 1e-6                               # no worse than the reference
        assert (y.detach().cpu().float() - case["y"].float()).abs().max() <= 2 ** -7 * case["y"].float().abs().max()
        assert (gi.float() - case["grad_input"].float()).abs().max() <= 2 ** -6 * case["grad_input"].float().abs().max()
    del w2


def test_forward_always_rescatters_without_the_fused_optimizer(api):
    """Reference semantics (smt.py:332-341): EVERY forward writes selected_weight into the dense weight.  Updates that
    bypass the Parameter's version counter - `p.data.add_()` (what DeepSpeed's FusedAdam does) or a write through a flat
    buffer that `p.data` aliases (BF16_Optimizer / ZeRO partitions) - must be visible in the next forward."""
    M, _H = api
    torch.manual_seed(0)
    w = torch.nn.Parameter(torch.randn(512, 512, device="cuda").bfloat16())
    layer = M.LinearLayer_MatrixSparsity(w, index_list=[(0, 1), (1, 0)])
    x = torch.randn(1, 8, 512, device="cuda").bfloat16()
    y0 = layer(x)
    w.data[0:256, 256:512] = 7.0                       # corrupt a selected block behind the module's back
    assert torch.equal(layer(x), y0)                   # the forward's scatter repairs it, like the reference's loop
    # (1) in-place update through .data: version counter does not move
    v0 = layer.selected_weight._version
    layer.selected_weight.data.add_(1.0)
    assert layer.selected_weight._version == v0
    y1 = layer(x)
    want = O.gather_blocks(w.detach().cpu(), layer.index_list, 256)
    assert torch.equal(want, layer.selected_weight.detach().cpu())          # dense weight now holds the update
    assert not torch.equal(y1, y0)
    # (2) .data re-pointed into a flat buffer, then the flat buffer is written (no version bump, same data_ptr)
    flat = torch.zeros(layer.selected_weight.numel() + 64, dtype=torch.bfloat16, device="cuda")
    view = flat[64:].view_as(layer.selected_weight)
    view.copy_(layer.selected_weight.data)
    layer.selected_weight.data = view
    flat.mul_(0.5)
    y2 = layer(x)
    assert torch.equal(O.gather_blocks(w.detach().cpu(), layer.index_list, 256), layer.selected_weight.detach().cpu())
    assert not torch.equal(y2, y1)
    # the channel-sparsity twin follows the same rule
    wc = torch.nn.Parameter(torch.randn(256, 512, device="cuda").bfloat16())
    ch = M.LinearLayer_ChannelSparsity(wc, index_list=[3, 500, 17])
    ch(x)
    ch.selected_weight.data.add_(1.0)
    ch(x)
    assert torch.equal(wc.detach()[:, [3, 500, 17]].t().contiguous(), ch.selected_weight.detach())


def test_fused_optimizer_skips_the_scatter_only_while_it_vouches_for_the_weight(api):
    """Under SMTAdam the dense blocks are written by the Adam kernel, so forward launches nothing - until anything
    invalidates that: a version-counted write to the Parameter, or `.data` being re-pointed elsewhere."""
    M, _H = api
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(1)
    w = torch.nn.Parameter(torch.randn(512, 512, device="cuda").bfloat16() * 0.05)
    layer = M.LinearLayer_MatrixSparsity(w, index_list=[(0, 1), (1, 0)])
    opt = SMTAdam([layer.selected_weight], lr=1e-2)
    x = torch.randn(2, 16, 512, device="cuda").bfloat16()
    opt.zero_grad()
    layer(x).float().pow(2).mean().backward()
    opt.step()
    assert torch.equal(O.gather_blocks(w.detach().cpu(), layer.index_list, 256), layer.selected_weight.detach().cpu())
    n0 = ops.LAUNCHES["total"]
    with torch.no_grad():
        layer(x)
        layer(x)
    assert ops.LAUNCHES["total"] == n0                 # no scatter launched: SMTAdam vouches for the dense weight
    with torch.no_grad():
        layer.selected_weight.mul_(2.0)                # version-counted write => mark invalid => scatter again
        layer(x)
    assert ops.LAUNCHES["total"] == n0 + 1
    assert torch.equal(O.gather_blocks(w.detach().cpu(), layer.index_list, 256), layer.selected_weight.detach().cpu())
    opt.zero_grad()
    layer(x).float().pow(2).mean().backward()
    opt.step()
    layer.selected_weight.data = layer.selected_weight.data.clone() * 3   # re-pointed storage => invalid
    n1 = ops.LAUNCHES["total"]
    with torch.no_grad():
        layer(x)
    assert ops.LAUNCHES["total"] == n1 + 1
    assert torch.equal(O.gather_blocks(w.detach().cpu(), layer.index_list, 256), layer.selected_weight.detach().cpu())


def test_convert_back_merges_blocks(api):
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=256, hidden_size=256, intermediate_size=512, num_hidden_layers=2,
                      num_attention_heads=4, num_key_value_heads=4, max_position_embeddings=64)
    model = LlamaForCausalLM(cfg).cuda().bfloat16()
    sel_attn = {("q_proj", 0): [(0, 0)], ("v_proj", 1): [(0, 0)]}
    sel_mlp = {("down_proj", 1): [(0, 1), (0, 0)]}
    M.freeze_unselected_matrix_layer(model, sel_mlp, sel_attn)
    M.convert_linear_layer_to_matrix_sparsity(model, sel_mlp, sel_attn)
    kinds = {n: type(m).__name__ for n, m in model.named_modules() if n.endswith(("_proj",))}
    assert kinds["model.layers.0.self_attn.q_proj"] == "LinearLayer_MatrixSparsity"
    assert kinds["model.layers.1.mlp.down_proj"] == "LinearLayer_MatrixSparsity"
    assert kinds["model.layers.0.self_attn.k_proj"] == "Linear"
    trainable = [n for n, p in model.named_parameters() if p.requires_grad]
    assert sorted(trainable) == sorted(["model.layers.0.self_attn.q_proj.selected_weight",
                                        "model.layers.1.self_attn.v_proj.selected_weight",
                                        "model.layers.1.mlp.down_proj.selected_weight"])
    q = model.model.layers[0].self_attn.q_proj
    with torch.no_grad():
        q.selected_weight.fill_(0.25)
    M.convert_matrix_sparsity_to_linear_layer(model)
    lin = model.model.layers[0].self_attn.q_proj
    assert type(lin) is torch.nn.Linear and lin.weight is q.weight
    assert (lin.weight[:256, :256] == 0.25).all()
    assert "selected_weight" not in "".join(model.state_dict().keys())


def test_config1_end_to_end_vs_reference_golden(api):
    """BASELINE config 1 (2-layer LLaMA, hidden 512, 256x256 blocks, 1 % q/k/v, fp32): warm-up capture ->
    selection -> freeze -> convert -> param groups -> clipped AdamW steps, against the reference's own run."""
    M, H = api
    from sparse_matrix_tuning_b200.optim import SMTAdam
    from sparse_matrix_tuning_b200.warmup import WarmupGradAccumulator
    gold = load_golden("config1_e2e.pt")
    c = GI.CONFIG1
    model, batches = GI.make_config1(device="cuda")
    named = list(model.named_parameters())
    dims = O.targeted_module_dims(named)
    n_attn = O.block_budget(named, c["attn_ratio"])
    assert dims == gold["dims"] and n_attn == gold["n_attn"]
    acc = WarmupGradAccumulator(block=256, mode="elementwise")
    for it in range(c["warmup_steps"]):
        model.zero_grad()
        out = model(input_ids=batches[it], labels=batches[it], use_cache=False)
        out.loss.backward()
        assert abs(out.loss.item() - gold["warm_losses"][it]) <= 5e-5
        acc.accumulate(model.named_parameters())
    model.zero_grad(set_to_none=True)
    sel = H.select_submatrix_based_on_grads(acc.grads(), dims, n_attn, selection_strategy="no_restriction")
    assert [(k, list(v)) for k, v in sel.items()] == [(k, [tuple(t) for t in v]) for k, v in gold["selection"]]
    model = M.freeze_unselected_matrix_layer(model, {}, sel)
    model = M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    assert [(n, tuple(p.shape)) for n, p in model.named_parameters() if p.requires_grad] == gold["trainable"]
    groups = M.get_optimizer_sparse_grouped_parameters(model, 0.0, c["smt_lr"])
    opt = SMTAdam(groups, lr=c["smt_lr"], betas=(0.9, 0.95), max_grad_norm=1.0)
    losses = []
    for it in range(c["sparse_steps"]):
        opt.zero_grad()
        b = batches[c["warmup_steps"] + it]
        out = model(input_ids=b, labels=b, use_cache=False)
        out.loss.backward()
        if it == 0:
            for n, p in model.named_parameters():
                if p.requires_grad:
                    ref = gold["first_grads"][n]
                    assert (p.grad.cpu() - ref).abs().max().item() <= 1e-4 * ref.abs().max().item() + 1e-9, n
            norm = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in model.parameters() if p.requires_grad)).item()
            assert abs(norm - gold["grad_norms"][0]) <= 1e-4 * gold["grad_norms"][0]
        opt.step()
        losses.append(out.loss.item())
    assert max(abs(a - b) for a, b in zip(losses, gold["losses"])) <= 5e-5, (losses, gold["losses"])
    # Adam normalises each element by sqrt(v): where a gradient is ~0 its SIGN decides a +-lr move, so elementwise
    # agreement is bounded by (#steps * lr) in the worst case and must be tight on average.
    for n, p in model.named_parameters():
        if p.requires_grad:
            d = (p.detach().cpu() - gold["final_selected"][n]).abs()
            assert d.max().item() <= 2 * c["sparse_steps"] * c["smt_lr"]
            assert d.mean().item() <= 2e-7, (n, d.mean().item())
    # the dense weights already hold the updated blocks (fused write-back): forward needs no scatter
    for mod in model.modules():
        if isinstance(mod, M.LinearLayer_MatrixSparsity):
            assert torch.equal(O.gather_blocks(mod.weight.detach().cpu(), mod.index_list, 256),
                               mod.selected_weight.detach().cpu())


def test_grouped_backward_equals_per_module_backward(api):
    """Deferring every module's block-gradient GEMM to one grouped launch at the end of the backward pass must not
    change the gradients, must be complete when loss.backward() returns, and must compose with checkpointing."""
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200.optim import SMTAdam

    def run(grouped, ckpt):
        torch.manual_seed(0)
        cfg = LlamaConfig(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=3,
                          num_attention_heads=8, num_key_value_heads=4, max_position_embeddings=128)
        model = LlamaForCausalLM(cfg).cuda().bfloat16()
        sel = {("q_proj", 0): [(0, 1), (1, 0)], ("k_proj", 0): [(0, 0)], ("v_proj", 1): [(0, 1)],
               ("q_proj", 2): [(1, 1), (0, 0), (0, 1)]}
        M.freeze_unselected_matrix_layer(model, {}, sel)
        M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
        if ckpt:
            model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
            model.enable_input_require_grads()
        model.train()
        opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-3), betas=(0.9, 0.95), max_grad_norm=1.0)
        M.set_grouped_backward(grouped)
        try:
            ids = torch.randint(0, 512, (2, 96), generator=torch.Generator().manual_seed(1)).cuda()
            opt.zero_grad()
            loss = model(input_ids=ids, labels=ids, use_cache=False).loss
            loss.backward()
            from sparse_matrix_tuning_b200.smt import smt as S
            assert len(S._pending) == 0                       # the engine callback already flushed the group
            grads = opt.flat_grads()[0].clone()
            opt.step()
            params = torch.cat([p.detach().reshape(-1).float() for g in opt.param_groups for p in g["params"]])
            return loss.item(), grads.float(), params
        finally:
            M.set_grouped_backward(False)

    l0, g0, p0 = run(False, False)
    for grouped, ckpt in ((True, False), (True, True)):
        l1, g1, p1 = run(grouped, ckpt)
        assert l1 == l0
        assert (g1 - g0).abs().max().item() <= 2 ** -7 * g0.abs().max().item()   # bf16 grads, different split-K plans
        assert (p1 - p0).abs().max().item() <= 2.1e-3                            # one Adam step of lr 1e-3 (sign flips of ~0 grads)


def test_merged_export_and_resume(api):
    """SURVEY §8f row 1: a merged HF-format state dict reproduces the SMT model's logits in an UNMODIFIED
    LlamaForCausalLM, and (index lists + compact params + optimizer state) round-trip for a bit-exact resume."""
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200 import checkpoint as CK
    from sparse_matrix_tuning_b200.optim import SMTAdam
    cfg = LlamaConfig(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=2,
                      num_attention_heads=8, num_key_value_heads=4, max_position_embeddings=128)
    sel = {("q_proj", 0): [(1, 0), (0, 1)], ("v_proj", 1): [(0, 1)]}

    def build():
        torch.manual_seed(3)
        model = LlamaForCausalLM(cfg).cuda().bfloat16()
        M.freeze_unselected_matrix_layer(model, {}, sel)
        M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
        opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-3), betas=(0.9, 0.95), max_grad_norm=1.0)
        return model, opt

    ids = torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(4)).cuda()

    def train(model, opt, steps):
        for _ in range(steps):
            opt.zero_grad()
            model(input_ids=ids, labels=ids, use_cache=False).loss.backward()
            opt.step()

    model, opt = build()
    train(model, opt, 2)
    merged = CK.merged_state_dict(model)
    assert not any(k.endswith("selected_weight") for k in merged)
    torch.manual_seed(99)
    plain = LlamaForCausalLM(cfg).cuda().bfloat16()
    plain.load_state_dict(merged)
    with torch.no_grad():
        assert torch.equal(plain(input_ids=ids).logits, model(input_ids=ids).logits)
    # resume: state saved after 2 steps, restored into a fresh conversion, one more step on both == identical
    state = CK.smt_state(model, opt)
    assert CK.selection_from_state(state) == ({}, {k: list(v) for k, v in sel.items()})
    model2, opt2 = build()
    CK.load_smt_state(model2, state, opt2)
    train(model, opt, 1)
    train(model2, opt2, 1)
    for (n1, p1), (n2, p2) in zip(model.named_parameters(), model2.named_parameters()):
        assert n1 == n2 and torch.equal(p1, p2), n1
    for a, b in zip(opt._arenas, opt2._arenas):
        assert torch.equal(a.master, b.master) and torch.equal(a.exp_avg, b.exp_avg) and torch.equal(a.exp_avg_sq, b.exp_avg_sq)


def test_warmup_hook_mode_matches_post_backward_sweep(api):
    """Grad-ready hooks (with immediate release of .grad) accumulate exactly what the reference's post-backward sweep
    (fine_tune.py:716-768) accumulates."""
    _M, H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200.warmup import WarmupGradAccumulator
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=2,
                      num_attention_heads=8, num_key_value_heads=4, max_position_embeddings=128)
    model = LlamaForCausalLM(cfg).cuda().bfloat16()
    ids = [torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(s)).cuda() for s in (1, 2)]
    sweep = WarmupGradAccumulator(block=256, mode="elementwise", mlp=True)
    for b in ids:
        model.zero_grad(set_to_none=True)
        model(input_ids=b, labels=b, use_cache=False).loss.backward()
        sweep.accumulate(model.named_parameters())
    hooked = WarmupGradAccumulator(block=256, mode="elementwise", mlp=True)
    hooked.attach(model, free_grads=True)
    for b in ids:
        model.zero_grad(set_to_none=True)
        model(input_ids=b, labels=b, use_cache=False).loss.backward()
    hooked.detach()
    assert set(sweep.grads()) == set(hooked.grads()) and len(sweep.grads()) == 2 * 6
    for k in sweep.grads():
        assert torch.equal(sweep.grads()[k], hooked.grads()[k]), k
    assert model.model.layers[0].self_attn.q_proj.weight.grad is None        # released by the hook
    assert model.model.layers[0].self_attn.o_proj.weight.grad is not None    # not a captured module


def test_linearz_layouts_and_direct_apply(api):
    """linearZ.apply called directly (as the reference's fwbwTest does, smt.py:865-903), 2-D and 4-D inputs, and a
    NON-contiguous grad_output (transposed producer) — all must give the dense-slice gradients."""
    M, _H = api
    torch.manual_seed(5)
    w = torch.nn.Parameter(torch.randn(512, 768, device="cuda").bfloat16() * 0.05)
    idx = [(1, 2), (0, 0), (1, 0)]
    layer = M.LinearLayer_MatrixSparsity(w, index_list=idx)
    for shape in ((40, 768), (2, 3, 8, 768), (3, 16, 768)):
        x = torch.randn(*shape, device="cuda").bfloat16().requires_grad_(True)
        layer.selected_weight.grad = None
        y = M.linearZ.apply(x, layer.selected_weight, idx, layer.weight)
        assert y.shape == shape[:-1] + (512,)
        g = torch.randn(512, x.numel() // 768, device="cuda").bfloat16().t().reshape(y.shape)   # non-contiguous rows
        assert not g.reshape(-1, 512).is_contiguous() or len(shape) > 2
        y.backward(g)
        x2, g2 = x.detach().reshape(-1, 768).float(), g.reshape(-1, 512).float()
        dense = g2.t() @ x2                                                               # full dW = dy^T x
        want = torch.cat([dense[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256] for r, c in idx])
        got = layer.selected_weight.grad.float()
        assert got.shape == (3 * 256, 256)
        assert (got - want).abs().max().item() <= 2 ** -7 * want.abs().max().item()
        assert (x.grad.float() - (g2 @ w.detach().float()).reshape(shape)).abs().max().item() <= \
            2 ** -6 * x.grad.float().abs().max().item()


def test_gradient_accumulation_over_micro_batches(api):
    """Two backward passes without zero_grad accumulate into the flat gradient buffer, like autograd does."""
    M, _H = api
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(6)
    w = torch.nn.Parameter(torch.randn(256, 512, device="cuda").bfloat16() * 0.05)
    layer = M.LinearLayer_MatrixSparsity(w, index_list=[(0, 1)])
    opt = SMTAdam([layer.selected_weight], lr=1e-3)
    xs = [torch.randn(2, 64, 512, device="cuda").bfloat16() for _ in range(2)]
    gs = [torch.randn(2, 64, 256, device="cuda").bfloat16() for _ in range(2)]
    opt.zero_grad()
    for x, g in zip(xs, gs):
        layer(x).backward(g)
    want = sum(g.reshape(-1, 256).float().t() @ x.reshape(-1, 512).float()[:, 256:512] for x, g in zip(xs, gs))
    got = layer.selected_weight.grad.float()
    assert layer.selected_weight.grad.data_ptr() == opt.flat_grads()[0].data_ptr()   # .grad IS the flat (NCCL) buffer
    assert (got - want).abs().max().item() <= 2 ** -6 * want.abs().max().item()
    # zero_grad() is lazy for block parameters: the next delivery OVERWRITES (no memset, no read-modify-write) ...
    opt.zero_grad()
    layer(xs[0]).backward(gs[0])
    want0 = gs[0].reshape(-1, 256).float().t() @ xs[0].reshape(-1, 512).float()[:, 256:512]
    assert (layer.selected_weight.grad.float() - want0).abs().max().item() <= 2 ** -7 * want0.abs().max().item()
    # ... and a step that received no gradient at all sees zeros, not last step's values
    opt.step()
    before = opt.state[layer.selected_weight]["master"].clone()
    m_before = opt.state[layer.selected_weight]["exp_avg"].clone()
    opt.zero_grad()
    opt.step()
    assert not opt.flat_grads()[0].any()
    assert torch.allclose(opt.state[layer.selected_weight]["exp_avg"], m_before * 0.9)   # g = 0: m <- beta1 * m
    assert not torch.equal(opt.state[layer.selected_weight]["master"], before)           # momentum still moves p


def test_gradients_dropped_behind_the_optimizers_back(api):
    """`model.zero_grad()` (set_to_none=True by default) and `p.grad = None` detach `.grad` from the flat arena.  The
    next backward must start from a clean slate (not accumulate onto last step's values) and re-attach the view;
    parameters that are not fed by linearZ (e.g. layer norms in mixture mode) get their fresh `.grad` copied in."""
    M, _H = api
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(9)
    w = torch.nn.Parameter(torch.randn(256, 512, device="cuda").bfloat16() * 0.05)
    layer = M.LinearLayer_MatrixSparsity(w, index_list=[(0, 1), (0, 0)])
    norm_w = torch.nn.Parameter(torch.ones(512, device="cuda").bfloat16())
    opt = SMTAdam([layer.selected_weight, norm_w], lr=1e-3)
    x = torch.randn(2, 64, 512, device="cuda").bfloat16()
    g = torch.randn(2, 64, 256, device="cuda").bfloat16()

    def fwd_bwd():
        layer(x * norm_w).backward(g)

    def truth():
        xx = (x * norm_w).reshape(-1, 512).float()
        full = g.reshape(-1, 256).float().t() @ xx
        return torch.cat([full[:, 256:512], full[:, 0:256]], 0)

    opt.zero_grad()
    fwd_bwd()
    g_norm_1 = norm_w.grad.detach().float().clone()
    opt.step()
    for p in (layer.selected_weight, norm_w):          # what HF Trainer / many loops do instead of opt.zero_grad()
        p.grad = None
    fwd_bwd()
    assert layer.selected_weight.grad is not None
    assert layer.selected_weight.grad.data_ptr() == opt.flat_grads()[0].data_ptr()
    want = truth()
    assert (layer.selected_weight.grad.float() - want).abs().max().item() <= 2 ** -7 * want.abs().max().item()
    assert norm_w.grad.data_ptr() != opt._arenas[0].grad_views[1].data_ptr()       # autograd made a fresh tensor
    fresh = norm_w.grad.detach().float().clone()
    opt.step()                                                                     # copies it in and re-attaches
    assert norm_w.grad.data_ptr() == opt._arenas[0].grad_views[1].data_ptr()
    assert torch.equal(norm_w.grad.float(), fresh)
    assert (fresh - g_norm_1).abs().max().item() <= 0.25 * g_norm_1.abs().max().item()          # one gradient, not two


def test_smtadam_unflattened_mode_matches_flat_mode(api):
    """`flatten=False` (a wrapper such as DeepSpeed owns the flat buffers; gradients arrive through autograd) must give
    the same parameters, masters and dense weights as the native flat arena."""
    M, _H = api
    from sparse_matrix_tuning_b200.optim import SMTAdam

    def run(flatten):
        torch.manual_seed(8)
        w1 = torch.nn.Parameter(torch.randn(512, 512, device="cuda").bfloat16() * 0.05)
        w2 = torch.nn.Parameter(torch.randn(256, 512, device="cuda").bfloat16() * 0.05)
        l1 = M.LinearLayer_MatrixSparsity(w1, index_list=[(0, 1), (1, 1)])
        l2 = M.LinearLayer_MatrixSparsity(w2, index_list=[(0, 0)])
        opt = SMTAdam([{"params": [l1.selected_weight, l2.selected_weight], "lr": 2e-3, "weight_decay": 0.01}],
                      betas=(0.9, 0.95), max_grad_norm=1.0, flatten=flatten)
        for step in range(3):
            g = torch.Generator(device="cuda").manual_seed(step)
            x = torch.randn(2, 32, 512, device="cuda", generator=g).bfloat16()
            opt.zero_grad()
            (l2(l1(x)).float().pow(2).mean()).backward()
            opt.step()
        masters = [opt.state[p]["master"].reshape(-1).clone() for p in (l1.selected_weight, l2.selected_weight)]
        return (l1.selected_weight.detach().clone(), l2.selected_weight.detach().clone(), w1.detach().clone(),
                w2.detach().clone(), masters)

    a, b = run(True), run(False)
    for t1, t2 in zip(a[:4], b[:4]):
        assert torch.equal(t1, t2)
    for m1, m2 in zip(a[4], b[4]):
        assert torch.equal(m1, m2)


def test_activation_capture_hooks_and_channel_selection(api):
    """fine_tune.py:586-708 restated: |x| of every Linear input accumulated over two batches, then
    select_channel_based_on_activation — device accumulators vs the oracle on the same activations."""
    _M, H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200.warmup import WarmupActivationAccumulator
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=512, hidden_size=256, intermediate_size=512, num_hidden_layers=2,
                      num_attention_heads=4, num_key_value_heads=4, max_position_embeddings=128)
    model = LlamaForCausalLM(cfg).cuda().bfloat16().eval()
    ids = [torch.randint(0, 512, (3, 40), generator=torch.Generator().manual_seed(s)).cuda() for s in (1, 2)]
    ref_acts = {}

    def ref_hook(key):
        def fn(_m, args):
            a = args[0].detach().abs().cpu().float()                     # fine_tune.py:651-671
            ref_acts[key] = a if key not in ref_acts else ref_acts[key] + a
        return fn

    acc = WarmupActivationAccumulator()
    acc.attach(model)
    handles = []
    for name, mod in model.named_modules():
        if isinstance(mod, torch.nn.Linear) and ".layers." in name:
            kind = name.split(".")[-1]
            handles.append(mod.register_forward_pre_hook(ref_hook((kind, int(name.split(".")[2])))))
    with torch.no_grad():
        for b in ids:
            model(input_ids=b, use_cache=False)
    acc.detach()
    for h in handles:
        h.remove()
    assert set(acc.activations()) == set(ref_acts) and len(ref_acts) == 2 * 7
    for k, a in ref_acts.items():
        assert torch.allclose(acc.activations()[k].cpu(), a.sum(0), rtol=1e-5, atol=1e-5), k
    for strategy in ("mean_abs", "L2"):
        want = O.select_channels(ref_acts, 24, "no_restriction", strategy)
        got = H.select_channel_based_on_activation(acc.activations(), n=24, calculate_strategy=strategy)
        assert {k: sorted(v) for k, v in got.items()} == {k: sorted(v) for k, v in want.items()}


def test_fused_and_separate_split_k_reduction_are_bit_identical(api, monkeypatch):
    """The in-kernel (cooperative) reduction and the separate reduce kernel sum the same partials in the same order."""
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(1)
    for b, T, n in ((256, 4096, 3), (256, 2048, 9), (128, 8192, 5), (64, 4096, 7)):
        x = torch.randn(T, 1024, device="cuda").bfloat16()
        dy = torch.randn(T, 1024, device="cuda").bfloat16()
        perm = torch.randperm((1024 // b) ** 2)[:n]
        rc = ops.make_block_rc([(int(p) // (1024 // b), int(p) % (1024 // b)) for p in perm], "cuda")
        assert ops.block_grad_gemm_plan(n, b, T, torch.bfloat16)[0] > 1
        monkeypatch.delenv("SMT_GEMM_NO_FUSED_REDUCE", raising=False)
        fused = [ops.block_grad_gemm(x, dy, rc, b, out_dtype=dt) for dt in (torch.float32, torch.bfloat16)]
        again = ops.block_grad_gemm(x, dy, rc, b, out_dtype=torch.float32)
        monkeypatch.setenv("SMT_GEMM_NO_FUSED_REDUCE", "1")
        plain = [ops.block_grad_gemm(x, dy, rc, b, out_dtype=dt) for dt in (torch.float32, torch.bfloat16)]
        monkeypatch.delenv("SMT_GEMM_NO_FUSED_REDUCE", raising=False)
        assert torch.equal(fused[0], plain[0]) and torch.equal(fused[1], plain[1]) and torch.equal(fused[0], again)
    # many back-to-back launches re-arm the arrival counters correctly, in the block-tile kernel and in the run-tile
    # kernel (b = 64 / 128; runs of 1 to 4 / 2 blocks), which calls the same fused reduction; launches interleaved
    runs = []
    for rb in (64, 128):
        nb = 1024 // rb
        idx = list(dict.fromkeys([(0, 3), (0, 1), (3, 0), (0, 0), (2, 2), (0, 2), (3, 3), (1, 1), (3, 1), (0, nb - 1)]))
        args = (x, dy, ops._runs_for(idx, rb, x.device), rb)
        assert ops.load().smt_block_grad_gemm_runs_workspace_bytes(args[2][1], rb, T) > 0          # split-K
        runs.append((args, ops._gemm_runs(*args, torch.empty((len(idx) * rb, rb), device="cuda"), False)))
    ref = ops.block_grad_gemm(x, dy, rc, b, out_dtype=torch.float32)
    for _ in range(50):
        assert torch.equal(ops.block_grad_gemm(x, dy, rc, b, out_dtype=torch.float32), ref)
        for args, want in runs:
            assert torch.equal(ops._gemm_runs(*args, torch.empty_like(want), False), want)


def test_config1_bf16_steady_state_vs_reference_golden(api):
    """BASELINE config 1 in bf16 (the training dtype): the reference's own bf16 SMT steps (CPU, fp32-master AdamW with
    clip 1.0) against SMTAdam + the tcgen05 block-gradient GEMM, with the reference's selection.
    Tolerances: losses 2e-2 abs (bf16 forward of a 32 000-way softmax on two different back ends), first-step block
    gradients 2^-6 of the tensor max, final compact weights within a few bf16 ulps of 0.02-scale weights."""
    M, _H = api
    from sparse_matrix_tuning_b200.optim import SMTAdam
    gold = load_golden("config1_bf16.pt")
    c = GI.CONFIG1
    sel = {k: [tuple(t) for t in v] for k, v in gold["selection"]}
    model, batches = GI.make_config1()
    model = model.to(torch.bfloat16).cuda()
    batches = [b.cuda() for b in batches]
    model = M.freeze_unselected_matrix_layer(model, {}, sel)
    model = M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, c["smt_lr"]), lr=c["smt_lr"], betas=(0.9, 0.95),
                  max_grad_norm=1.0)
    M.set_grouped_backward(True)
    try:
        losses = []
        for it in range(c["sparse_steps"]):
            opt.zero_grad()
            b = batches[c["warmup_steps"] + it]
            out = model(input_ids=b, labels=b, use_cache=False)
            out.loss.backward()
            if it == 0:
                for n, p in model.named_parameters():
                    if p.requires_grad:
                        ref = gold["first_grads"][n].float()
                        assert (p.grad.float().cpu() - ref).abs().max().item() <= 2 ** -6 * ref.abs().max().item(), n
            opt.step()
            losses.append(out.loss.item())
    finally:
        M.set_grouped_backward(False)
    assert max(abs(a - b) for a, b in zip(losses, gold["losses"])) <= 2e-2, (losses, gold["losses"])
    for n, p in model.named_parameters():
        if p.requires_grad:
            d = (p.detach().float().cpu() - gold["final_selected"][n].float()).abs()
            assert d.max().item() <= 2 * c["sparse_steps"] * c["smt_lr"] + 2 ** -8 * 0.1, (n, d.max().item())
            assert d.mean().item() <= 4e-5, (n, d.mean().item())


def test_edge_cases_empty_index_list_frozen_compact_and_oversized_n(api):
    M, H = api
    torch.manual_seed(9)
    w = torch.nn.Parameter(torch.randn(256, 512, device="cuda").bfloat16() * 0.05)
    # (a) a module converted with NO selected block behaves like a frozen dense layer (reference: empty [0, 256] param)
    empty = M.LinearLayer_MatrixSparsity(w, index_list=[])
    assert tuple(empty.selected_weight.shape) == (0, 256)
    x = torch.randn(2, 8, 512, device="cuda").bfloat16().requires_grad_(True)
    y = empty(x)
    y.sum().backward()
    assert torch.equal(y, torch.matmul(x.detach(), w.t())) and x.grad is not None
    assert empty.selected_weight.grad is None or empty.selected_weight.grad.numel() == 0
    # (b) frozen compact parameter: no block-gradient work, input gradient still flows
    layer = M.LinearLayer_MatrixSparsity(w, index_list=[(0, 1)])
    layer.selected_weight.requires_grad = False
    x2 = torch.randn(2, 8, 512, device="cuda").bfloat16().requires_grad_(True)
    layer(x2).sum().backward()
    assert layer.selected_weight.grad is None and x2.grad is not None
    # (c) n larger than what exists: everything comes back, best first (smt_helper.py:111-119 never pops)
    grads = {("q_proj", 0): torch.randn(512, 512), ("k_proj", 3): torch.randn(256, 512)}
    dims = {"q_proj": [512, 512], "k_proj": [256, 512]}
    for strat in ("no_restriction", "norm_dist"):
        got = H.select_submatrix_based_on_grads(grads, dims, 1000, selection_strategy=strat)
        want = O.select_submatrix(grads, dims, 1000, strat)
        assert {k: sorted(v) for k, v in got.items()} == {k: sorted(v) for k, v in want.items()}
        assert sum(len(v) for v in got.values()) == 6
    act = {("q_proj", 0): torch.rand(2, 16, 64), ("up_proj", 1): torch.rand(2, 16, 32)}
    got = H.select_channel_based_on_activation(act, n=500)
    assert sorted(got[("q_proj", 0)]) == list(range(64)) and sorted(got[("up_proj", 1)]) == list(range(32))
    assert list(got.items()) == [(k, list(v)) for k, v in O.select_channels(act, 500).items()]


def test_mixture_mode_conversion(api):
    """mixture=True (fine_tune.py --no_limit_mixture): attention modules are looked up in the FIRST dict and o_proj may
    be selected too (smt.py:146-176, 657-678)."""
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=256, hidden_size=256, intermediate_size=512, num_hidden_layers=2,
                      num_attention_heads=4, num_key_value_heads=4, max_position_embeddings=64)
    model = LlamaForCausalLM(cfg).cuda().bfloat16()
    sel = {("o_proj", 1): [(0, 0)], ("k_proj", 0): [(0, 0)], ("gate_proj", 1): [(1, 0), (0, 0)]}
    M.freeze_unselected_matrix_layer(model, sel, {}, mixture=True)
    M.convert_linear_layer_to_matrix_sparsity(model, sel, {}, mixture=True)
    converted = sorted(n for n, m in model.named_modules() if isinstance(m, M.LinearLayer_MatrixSparsity))
    assert converted == ["model.layers.0.self_attn.k_proj", "model.layers.1.mlp.gate_proj", "model.layers.1.self_attn.o_proj"]
    assert sorted(n for n, p in model.named_parameters() if p.requires_grad) == sorted(c + ".selected_weight" for c in converted)
    ids = torch.randint(0, 256, (2, 32), device="cuda")
    model(input_ids=ids, labels=ids, use_cache=False).loss.backward()
    g = model.model.layers[1].mlp.gate_proj.selected_weight.grad
    assert g is not None and tuple(g.shape) == (512, 256) and g.abs().sum() > 0


@pytest.mark.parametrize("case", load_golden("linearchannel_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_linear_layer_channel_sparsity_golden(api, case):
    """Square weights = the shapes the reference's channel layer runs on: y, grad_input and the [n, out] channel
    gradient must match the reference's outputs; the compact parameter holds the selected COLUMNS."""
    M, _H = api
    spec = case["spec"]
    x, dy, w, idx = case["x"], case["dy"], case["w"], case["index_list"]
    layer = M.LinearLayer_ChannelSparsity(torch.nn.Parameter(w.clone().cuda()), bias=None, index_list=idx)
    assert torch.equal(layer.selected_weight.detach().cpu(), O.gather_columns(w, idx))       # gather: exact
    assert layer.selected_weight.requires_grad and not layer.weight.requires_grad
    xin = x.clone().cuda().requires_grad_(True)
    y = layer(xin)
    y.backward(dy.cuda())
    gw, gi = layer.selected_weight.grad.cpu(), xin.grad.cpu()
    assert gw.shape == case["grad_weight"].shape and gw.dtype == case["grad_weight"].dtype
    truth = x.reshape(-1, x.shape[-1])[:, idx].double().t() @ dy.reshape(-1, dy.shape[-1]).double()
    scale = truth.abs().max().item()
    if spec["dtype"] == "float32":
        assert (gw - case["grad_weight"]).abs().max().item() <= 1e-5 * scale
        assert torch.allclose(y.detach().cpu(), case["y"], rtol=1e-4, atol=1e-5)
        assert torch.allclose(gi, case["grad_input"], rtol=1e-4, atol=1e-5)
    else:
        err = (gw.double() - truth).abs().max().item() / scale
        ref_err = (case["grad_weight"].double() - truth).abs().max().item() / scale
        assert err <= 2 ** -7 and err <= ref_err * 1.10 + 1e-6                               # no worse than the reference
        assert (y.detach().cpu().float() - case["y"].float()).abs().max() <= 2 ** -7 * case["y"].float().abs().max()
        assert (gi.float() - case["grad_input"].float()).abs().max() <= 2 ** -6 * case["grad_input"].float().abs().max()


def test_channel_sparsity_non_square_training_and_merge(api):
    """What the reference cannot do: a 384 x 640 weight.  Column gather / scatter are exact against the oracle's
    column restatement, the gradient matches it, SMTAdam updates only the selected columns and the write-back lands
    before the next forward; convert_channel_sparsity_to_linear_layer merges."""
    M, _H = api
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(7)
    B, S, fin, fout = 3, 50, 640, 384
    idx = [639, 0, 5, 64, 63, 320, 17]
    w = (torch.randn(fout, fin) * 0.05).bfloat16()
    x = torch.randn(B, S, fin).bfloat16()
    dy = torch.randn(B, S, fout).bfloat16()

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.layers = torch.nn.ModuleList([torch.nn.Linear(fin, fout, bias=False)])

    net = Net().cuda().bfloat16()
    with torch.no_grad():
        net.layers[0].weight.copy_(w.cuda())
    layer = M.LinearLayer_ChannelSparsity(net.layers[0].weight, bias=None, index_list=idx)
    net.layers[0] = layer
    assert torch.equal(layer.selected_weight.detach().cpu(), O.gather_columns(w, idx))
    opt = SMTAdam([layer.selected_weight], lr=1e-2, betas=(0.9, 0.95), max_grad_norm=1.0)
    xin = x.cuda().requires_grad_(True)
    y = layer(xin)
    y.backward(dy.cuda())
    gi_ref, gw_ref = O.linearchannel_backward(x.float(), dy.float(), w.float(), idx)
    scale = gw_ref.abs().max().item()
    assert (layer.selected_weight.grad.float().cpu() - gw_ref).abs().max().item() <= 2 ** -7 * scale
    assert (xin.grad.float().cpu() - gi_ref).abs().max().item() <= 2 ** -6 * gi_ref.abs().max().item()
    before = layer.weight.detach().clone()
    opt.step()
    y2 = layer(x.cuda())                                            # forward re-scatters the updated columns
    after = layer.weight.detach()
    keep = [c for c in range(fin) if c not in idx]
    assert torch.equal(after[:, keep], before[:, keep])             # untouched columns are bit-identical
    assert torch.equal(after[:, idx].t().contiguous(), layer.selected_weight.detach())
    assert not torch.equal(after[:, idx], before[:, idx])
    assert torch.equal(y2, torch.matmul(x.cuda(), after.t()))
    M.convert_channel_sparsity_to_linear_layer(net, part_module_name=['layers'])
    assert isinstance(net.layers[0], torch.nn.Linear) and net.layers[0].weight.data_ptr() == after.data_ptr()


def test_channel_freeze_and_convert_on_tiny_llama(api):
    """fine_tune.py:511-520: freeze_unselected_channel_layer + convert_linear_layer_to_channel_sparsity on a tiny
    LLaMA (rectangular k/v and MLP weights included); one training step decreases nothing it should not touch."""
    M, H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, vocab_size=256)
    torch.manual_seed(0)
    model = LlamaForCausalLM(cfg).cuda()
    sel_mlp = {("gate_proj", 0): [1, 2, 100], ("down_proj", 1): [3, 255]}
    sel_attn = {("q_proj", 1): [5, 6], ("v_proj", 0): [0, 127]}
    model = M.freeze_unselected_channel_layer(model, sel_mlp, sel_attn)
    model = M.convert_linear_layer_to_channel_sparsity(model, sel_mlp, sel_attn)
    converted = {n for n, m in model.named_modules() if isinstance(m, M.LinearLayer_ChannelSparsity)}
    assert converted == {"model.layers.0.mlp.gate_proj", "model.layers.1.mlp.down_proj",
                         "model.layers.1.self_attn.q_proj", "model.layers.0.self_attn.v_proj"}
    trainable = {n: p for n, p in model.named_parameters() if p.requires_grad}
    assert all(n.endswith("selected_weight") for n in trainable) and len(trainable) == 4
    assert trainable["model.layers.0.self_attn.v_proj.selected_weight"].shape == (2, 64)     # [n, out_features]
    assert trainable["model.layers.1.mlp.down_proj.selected_weight"].shape == (2, 128)
    groups = M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-3)
    opt = torch.optim.AdamW(groups, lr=1e-3)
    ids = torch.randint(0, 256, (2, 16), device="cuda")
    losses = []
    for _ in range(3):
        out = model(input_ids=ids, labels=ids)
        out.loss.backward()
        opt.step(); opt.zero_grad()
        losses.append(out.loss.item())
    assert losses[-1] < losses[0]


def test_channel_modules_in_merged_export_and_resume(api):
    """checkpoint.py treats channel-sparse modules like block-sparse ones: the merged state dict has the trained columns
    written back and no `selected_weight` keys; smt_state / load_smt_state round-trip the compact parameter."""
    M, _H = api
    from sparse_matrix_tuning_b200 import checkpoint as CK

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.layers = torch.nn.ModuleList([torch.nn.Linear(192, 320, bias=False), torch.nn.Linear(320, 64, bias=False)])

    torch.manual_seed(3)
    net = Net().cuda().bfloat16()
    idx = [5, 191, 64]
    net.layers[0] = M.LinearLayer_ChannelSparsity(net.layers[0].weight, bias=None, index_list=idx)
    layer = net.layers[0]
    w0 = layer.weight.detach().clone()
    with torch.no_grad():
        layer.selected_weight.add_(1.0)
    merged = CK.merged_state_dict(net)
    assert set(merged) == {"layers.0.weight", "layers.1.weight"}
    assert torch.equal(merged["layers.0.weight"][:, idx].t().contiguous(), layer.selected_weight.detach())
    keep = [c for c in range(192) if c not in idx]
    assert torch.equal(merged["layers.0.weight"][:, keep], w0[:, keep])
    state = CK.smt_state(net)
    assert state["index_lists"]["layers.0"] == idx and state["block"]["layers.0"] is None
    with torch.no_grad():
        layer.selected_weight.zero_()
    CK.load_smt_state(net, state)
    assert torch.equal(layer.selected_weight.detach(), state["selected_weight"]["layers.0"])
    assert torch.equal(layer.weight[:, idx].t().contiguous(), layer.selected_weight.detach())


def test_smtadam_under_the_drivers_lr_scheduler(api):
    """fine_tune.py:367-373: the SMT phase builds `get_scheduler("linear", optimizer, num_warmup_steps=smt_lr_warmup_steps,
    num_training_steps=...)` over the new optimizer; group 0's lr starts from smt_lr (smt.py:517-518 overrides the
    optimizer's lr).  SMTAdam must follow the schedule exactly like torch.optim.AdamW on fp32 copies of the same blocks."""
    M, _H = api
    from transformers import get_scheduler
    from sparse_matrix_tuning_b200.optim import SMTAdam
    torch.manual_seed(12)
    w = torch.nn.Parameter(torch.randn(512, 512, device="cuda") * 0.05)            # fp32: masters == parameters
    layer = M.LinearLayer_MatrixSparsity(w, index_list=[(1, 0), (0, 1)])
    holder = torch.nn.Module()
    holder.layer = layer
    groups = M.get_optimizer_sparse_grouped_parameters(holder, 0.0, 3e-4)
    opt = SMTAdam(groups, lr=9.65e-6, betas=(0.9, 0.95))                            # fine_tune.py:352-363
    sched = get_scheduler(name="linear", optimizer=opt, num_warmup_steps=3, num_training_steps=10)
    ref_p = torch.nn.Parameter(layer.selected_weight.detach().clone())
    ref_opt = torch.optim.AdamW([{"params": [ref_p], "lr": 3e-4, "weight_decay": 0.0}], lr=9.65e-6, betas=(0.9, 0.95),
                                eps=1e-8)
    ref_sched = get_scheduler(name="linear", optimizer=ref_opt, num_warmup_steps=3, num_training_steps=10)
    lrs = []
    for step in range(8):
        g = torch.Generator(device="cuda").manual_seed(step)
        x = torch.randn(2, 32, 512, device="cuda", generator=g)
        dy = torch.randn(2, 32, 512, device="cuda", generator=g)
        opt.zero_grad()
        layer(x).backward(dy)
        ref_p.grad = layer.selected_weight.grad.detach().clone()
        opt.step()
        sched.step()
        ref_opt.step()
        ref_sched.step()
        lrs.append(opt.param_groups[0]["lr"])
        assert opt.param_groups[0]["lr"] == ref_opt.param_groups[0]["lr"]
        assert (layer.selected_weight.detach() - ref_p.detach()).abs().max().item() <= 2e-6 * (step + 1)
    assert lrs[0] == pytest.approx(3e-4 / 3) and lrs[2] == pytest.approx(3e-4) and lrs[-1] < lrs[3]   # warm-up, then decay
    assert torch.equal(O.gather_blocks(w.detach().cpu(), layer.index_list, 256), layer.selected_weight.detach().cpu())


@pytest.mark.parametrize("n,out_f,T,dtype", [(1, 1024, 300, torch.bfloat16), (5, 4096, 1000, torch.bfloat16),
                                              (100, 1024, 2048, torch.float16), (130, 14336, 777, torch.bfloat16),
                                              (64, 512, 64, torch.bfloat16)])
def test_channel_grad_gemm_vs_fp32_matmul(api, n, out_f, T, dtype):
    """The channel-sparsity weight gradient `partial_input^T @ grad_output` (smt.py:283-284) on the tcgen05 pipeline:
    packed channels padded by TMA zero fill, tiles stored with the row pitch of the [n, out] result.  fp32 accumulation,
    one rounding: within 2^-8 of the tensor max of the fp32 product (half an ulp of the largest element)."""
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(n)
    x = torch.randn(T, 2048, device="cuda").to(dtype)
    dy = torch.randn(T, out_f, device="cuda").to(dtype)
    idx_list = torch.randperm(2048)[:n].tolist()
    idx = ops.make_channel_idx(idx_list, "cuda", pad_to=8)
    partial = ops.channel_gather(x, idx)
    assert partial.shape == (T, (n + 7) // 8 * 8)
    assert torch.equal(partial[:, :n], x[:, idx_list]) and not partial[:, n:].any()
    got = ops.channel_grad_gemm(partial, n, dy)
    want = x[:, idx_list].float().t() @ dy.float()
    assert got.shape == (n, out_f) and got.dtype == dtype
    assert (got.float() - want).abs().max().item() <= 2 ** -8 * want.abs().max().item()
    assert torch.equal(got, ops.channel_grad_gemm(partial, n, dy))            # deterministic


def test_activation_based_block_selection_extension(api):
    """Block scores from activations (extension, parity unpinned): block column score = sum of its channels' scores
    (channel scores pinned by the reference goldens), same for every block row; top-n by the shared tie rule."""
    M, H = api
    torch.manual_seed(4)
    b = 256
    act = {("q_proj", 0): torch.rand(2, 16, 1024), ("k_proj", 0): torch.rand(2, 16, 1024), ("down_proj", 1): torch.rand(2, 16, 512)}
    act[("k_proj", 0)][:, :, 256:512] += 5.0                                   # plant one hot block column
    dims = {"q_proj": [1024, 1024], "k_proj": [512, 1024], "down_proj": [1024, 512]}
    sel = H.select_submatrix_based_on_activation(act, dims, 3)
    # the planted column outranks everything; with equal scores in a column the tie rule prefers the larger (i, j) tuple
    assert sel[("k_proj", 0)][:2] == [(1, 1), (0, 1)]
    want = {}
    for key, a in act.items():
        cs = O.channel_scores(a, "mean_abs")
        per_col = cs.view(-1, b).sum(1)
        rows = dims[key[0]][0] // b
        want[key] = per_col.unsqueeze(0).expand(rows, -1).contiguous()
    ref = O.select_from_scores(want, 3)
    assert {k: v for k, v in sel.items()} == {k: v for k, v in ref.items()}


@pytest.mark.parametrize("ckpt,grouped", [(False, False), (True, True)])
def test_fused_qkv_projections_match_the_unfused_model(api, ckpt, grouped):
    """f-2: `fuse_qkv_projections` must not change what the model computes: same loss, same compact gradients, same
    parameters after a step - with sparse and frozen members mixed, under checkpointing and grouped block gradients."""
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200.optim import SMTAdam

    def run(fuse):
        torch.manual_seed(0)
        cfg = LlamaConfig(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=3,
                          num_attention_heads=8, num_key_value_heads=4, max_position_embeddings=128)
        model = LlamaForCausalLM(cfg).cuda().bfloat16()
        sel = {("q_proj", 0): [(0, 1), (1, 0)], ("k_proj", 0): [(0, 0)], ("v_proj", 0): [(0, 1)],
               ("v_proj", 1): [(0, 0)], ("q_proj", 2): [(1, 1), (0, 0), (0, 1)]}      # layer 1: only v is sparse
        M.freeze_unselected_matrix_layer(model, {}, sel)
        M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
        if ckpt:
            model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
            model.enable_input_require_grads()
        model.train()
        n_fused = M.fuse_qkv_projections(model) if fuse else 0
        opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-3), betas=(0.9, 0.95), max_grad_norm=1.0)
        M.set_grouped_backward(grouped)
        try:
            ids = torch.randint(0, 512, (2, 96), generator=torch.Generator().manual_seed(1)).cuda()
            losses = []
            for _ in range(2):
                opt.zero_grad()
                n0 = ops.LAUNCHES["total"]
                loss = model(input_ids=ids, labels=ids, use_cache=False).loss
                loss.backward()
                launches = ops.LAUNCHES["total"] - n0
                grads = opt.flat_grads()[0].float().clone()
                opt.step()
                losses.append(loss.item())
            params = torch.cat([p.detach().reshape(-1).float() for g in opt.param_groups for p in g["params"]])
            names = sorted(k for k in model.state_dict().keys())
            return losses, grads, params, n_fused, launches, names
        finally:
            M.set_grouped_backward(False)
            M.unfuse_qkv_projections(model)

    l0, g0, p0, _, _, names0 = run(False)
    l1, g1, p1, n_fused, launches, names1 = run(True)
    assert n_fused == 3 and names0 == names1                        # every layer fused; state dict keys untouched
    assert launches >= 3 * (2 if ckpt else 1) + 3                   # fused forward (x2 with recomputation) + fused dgrad
    assert abs(l1[0] - l0[0]) <= 2e-2 and abs(l1[1] - l0[1]) <= 2e-2   # bf16 logits: one rounding vs the library's
    assert (g1 - g0).abs().max().item() <= 0.05 * g0.abs().max().item()
    assert (p1 - p0).abs().max().item() <= 2.1e-3 * 2               # two Adam steps of lr 1e-3


def test_fused_qkv_falls_back_when_called_out_of_pattern(api):
    """k_proj called with a different tensor, or alone, must give its own x @ Wk^T (no stale slice of a fused call)."""
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(3)
    cfg = LlamaConfig(vocab_size=256, hidden_size=512, intermediate_size=1024, num_hidden_layers=1,
                      num_attention_heads=8, num_key_value_heads=4, max_position_embeddings=64)
    model = LlamaForCausalLM(cfg).cuda().bfloat16()
    M.freeze_unselected_matrix_layer(model, {}, {})
    assert M.fuse_qkv_projections(model) == 1
    attn = model.model.layers[0].self_attn
    x = torch.randn(2, 16, 512, device="cuda").bfloat16()
    x_other = torch.randn(2, 16, 512, device="cuda").bfloat16()
    with torch.no_grad():
        q = attn.q_proj(x)                                   # fused call: k and v slices are cached for `x`
        k_other = attn.k_proj(x_other)                       # different tensor: plain path
        k = attn.k_proj(x)                                   # the cached slice
        v_alone = attn.v_proj(x_other)
    ref = lambda t, w: (t.float() @ w.float().t())
    tol = 2 ** -7
    for got, want in ((q, ref(x, attn.q_proj.weight)), (k, ref(x, attn.k_proj.weight)),
                      (k_other, ref(x_other, attn.k_proj.weight)), (v_alone, ref(x_other, attn.v_proj.weight))):
        assert (got.float() - want).abs().max().item() <= tol * want.abs().max().item()
    assert M.unfuse_qkv_projections(model) == 1 and "forward" not in attn.q_proj.__dict__


def test_chunked_flush_and_overlapped_exchange_on_one_gpu(api):
    """The data-parallel step's machinery with a world of one: the grouped block-gradient GEMM flushed in chunks DURING
    backward (layer boundaries, chunk_blocks pending), every chunk handed to `OverlappedGradExchange` (side stream, per-chunk
    sums of squares), the optimizer clipping with those partial norms.  Must equal the unchunked, exchange-free step."""
    M, _H = api
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200 import dp
    from sparse_matrix_tuning_b200.optim import SMTAdam

    def run(chunked):
        torch.manual_seed(0)
        cfg = LlamaConfig(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=4,
                          num_attention_heads=8, num_key_value_heads=4, max_position_embeddings=128)
        model = LlamaForCausalLM(cfg).cuda().bfloat16()
        sel = {("q_proj", 0): [(0, 1), (1, 0)], ("k_proj", 0): [(0, 0)], ("v_proj", 1): [(0, 1)],
               ("q_proj", 2): [(1, 1), (0, 0), (0, 1)], ("k_proj", 3): [(0, 1)], ("q_proj", 3): [(1, 0)]}
        M.freeze_unselected_matrix_layer(model, {}, sel)
        M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
        model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
        model.enable_input_require_grads()
        model.train()
        opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-3), betas=(0.9, 0.95), max_grad_norm=0.05)
        M.set_grouped_backward(True, chunk_blocks=2 if chunked else 0)
        ex = dp.OverlappedGradExchange(opt, sqnorm=True) if chunked else None
        try:
            ids = torch.randint(0, 512, (2, 96), generator=torch.Generator().manual_seed(1)).cuda()
            chunks = []
            if ex is not None:
                M.add_flush_listener(lambda sinks: chunks.append(len(sinks)))
            for it in range(2):
                opt.zero_grad()
                model(input_ids=ids, labels=ids, use_cache=False).loss.backward()
                if ex is not None and it == 0:
                    ex.finish()
                    ex.finish()                                    # idempotent: joining twice reduces nothing twice
                    assert opt._arenas[0].sq_override is not None and opt._arenas[0].sq_override.numel() >= 2
                grads = opt.flat_grads()[0].float().clone()
                opt.step()                                         # (second iteration: step() joins the exchange itself)
                src = opt.sqnorm_source
            params = torch.cat([p.detach().reshape(-1).float() for g in opt.param_groups for p in g["params"]])
            return grads, params, src, chunks
        finally:
            if ex is not None:
                ex.close()
            M._flush_listeners.clear()
            M.set_grouped_backward(False)

    g0, p0, src0, _ = run(False)
    g1, p1, src1, chunks = run(True)
    assert src1 == "partials" and len(chunks) >= 4 and max(chunks) <= 4          # several flushes per backward pass
    assert (g1 - g0).abs().max().item() <= 2 ** -7 * g0.abs().max().item()
    assert (p1 - p0).abs().max().item() <= 2.1e-3 * 2                             # clip active (max_norm 0.05): same norm


def test_many_small_blocks_through_the_api_use_run_tiles_and_match_the_reference_loop(api, monkeypatch):
    """b = 64 with every block of a 1024 x 1024 weight selected (256 blocks, 16 per block row): `linearZ.backward` takes
    the strip-sharing run kernel on its own (per-module launch) and must still reproduce the reference's per-block loop
    (oracle.linearz_backward restates smt.py:376-413) - no worse than the reference's own bf16 error vs fp64 truth."""
    M, _H = api
    from sparse_matrix_tuning_b200 import ops
    monkeypatch.setattr(M, "Block_dimension", 64)
    torch.manual_seed(2)
    b, nb = 64, 16
    idx = [(r, c) for r in range(nb) for c in range(nb)]
    torch.Generator().manual_seed(0)
    perm = torch.randperm(len(idx)).tolist()
    idx = [idx[i] for i in perm]                                   # list order = compact row order, not sorted
    w = (torch.randn(1024, 1024) * 0.02).bfloat16()
    x = torch.randn(2, 256, 1024).bfloat16()
    dy = torch.randn(2, 256, 1024).bfloat16()
    layer = M.LinearLayer_MatrixSparsity(torch.nn.Parameter(w.clone().cuda()), index_list=idx)
    xin = x.cuda().requires_grad_(True)
    layer(xin).backward(dy.cuda())
    assert ops.LAST_SINGLE["kernel"] == "runs"
    got = layer.selected_weight.grad.detach().cpu()
    truth = O.block_grad_truth(x, dy, idx, b)
    _gi, ref = O.linearz_backward(x, dy, w, idx, b)
    scale = truth.abs().max().item()
    err = (got.double() - truth).abs().max().item() / scale
    ref_err = (ref.double() - truth).abs().max().item() / scale
    assert err <= 2 ** -7 and err <= ref_err * 1.10 + 1e-6, (err, ref_err)
    assert (xin.grad.float().cpu() - _gi.float()).abs().max().item() <= 2 ** -6 * _gi.float().abs().max().item()
