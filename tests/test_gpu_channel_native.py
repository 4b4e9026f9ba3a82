"""Channel sparsity on the native training step: channel gradients delivered into the SMTAdam arena by the grouped
block-gradient launch (with per-tile sums of squares), the fused Adam step with its column write-back
(`smt_compact_adam_columns`), and channel q/k/v members in the fused projection group with the decoder-layer kernels."""
import copy

import numpy as np
import pytest
import torch

from oracle import smt_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def M(built_library):
    from sparse_matrix_tuning_b200.smt import smt
    return smt


@pytest.fixture
def grouped(M):
    M.set_grouped_backward(True)
    yield
    M.set_grouped_backward(False)


def _tiny_cfg(**kw):
    from transformers import LlamaConfig
    base = dict(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
                num_key_value_heads=2, head_dim=128, max_position_embeddings=256, attn_implementation="sdpa")
    base.update(kw)
    return LlamaConfig(**base)


def _channels(n, width, seed):
    return torch.randperm(width, generator=torch.Generator().manual_seed(seed))[:n].tolist()


# channel counts that are not multiples of 8 or of the tile (q: 4 row tiles of 64 at b = 128 -> 2 tiles, padded)
SEL_ATTN = {("q_proj", 0): _channels(77, 512, 1), ("k_proj", 0): _channels(5, 512, 2), ("v_proj", 0): _channels(130, 512, 3),
            ("q_proj", 1): _channels(64, 512, 4), ("v_proj", 1): _channels(13, 512, 5)}
SEL_MLP = {("gate_proj", 0): _channels(29, 512, 6), ("up_proj", 1): _channels(70, 512, 7),
           ("down_proj", 0): _channels(131, 1024, 8)}


def _model(M, sel_mlp, sel_attn, fuse):
    from transformers import LlamaForCausalLM
    torch.manual_seed(0)
    model = LlamaForCausalLM(_tiny_cfg()).cuda().bfloat16()
    M.freeze_unselected_channel_layer(model, sel_mlp, sel_attn)
    M.convert_linear_layer_to_channel_sparsity(model, sel_mlp, sel_attn)
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    model.train()
    if fuse:
        assert M.fuse_qkv_projections(model) == 2
        assert "forward" in model.model.layers[0].__dict__ and "forward" in model.model.norm.__dict__
    return model


def _train(M, native, sel_mlp, sel_attn, steps=3, lr=1e-3, monkeypatch=None):
    from sparse_matrix_tuning_b200.optim import SMTAdam
    if not native:      # the per-module path: no owner, so no sink, per-parameter Adam and a scatter on every forward
        monkeypatch.setattr(M.LinearLayer_ChannelSparsity, "_arena_ok", lambda self: False)
    model = _model(M, sel_mlp, sel_attn, fuse=native)
    opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, lr), betas=(0.9, 0.95), max_grad_norm=1.0)
    M.set_grouped_backward(native)
    try:
        gen = torch.Generator().manual_seed(1)
        losses, sources = [], []
        for _ in range(steps):
            ids = torch.randint(0, 512, (2, 128), generator=gen).cuda()
            opt.zero_grad()
            loss = model(input_ids=ids, labels=ids, use_cache=False).loss
            loss.backward()
            opt.step()
            losses.append(loss.item())
            sources.append(opt.sqnorm_source)
        params = torch.cat([opt.state[p]["master"].reshape(-1) for g in opt.param_groups for p in g["params"]])
        dense = torch.cat([m.weight.detach().reshape(-1).float() for m in model.modules()
                           if isinstance(m, M.LinearLayer_ChannelSparsity)])
        return losses, params, dense, sources, model, opt
    finally:
        M.set_grouped_backward(False)
        if not native:
            monkeypatch.undo()


@pytest.mark.parametrize("with_mlp", [False, True])
def test_native_channel_training_matches_the_per_module_path(M, monkeypatch, with_mlp):
    sel_mlp = SEL_MLP if with_mlp else {}
    steps, lr = 3, 1e-3
    l0, p0, d0, _s0, _m0, _o0 = _train(M, False, sel_mlp, SEL_ATTN, steps, lr, monkeypatch)
    l1, p1, d1, s1, model, opt = _train(M, True, sel_mlp, SEL_ATTN, steps, lr)
    assert max(abs(a - b) for a, b in zip(l0, l1)) <= 1e-2, (l0, l1)
    assert (p1 - p0).abs().max().item() <= 2 * steps * lr
    assert (d1 - d0).abs().max().item() <= 2 * steps * lr + 2 ** -6           # trained columns in the dense weights
    arena = opt._arenas[0]
    assert arena.all_sinks and arena.fused_writeback() is not None and "columns" in arena.fused_writeback()
    assert s1[-1] == "partials"                                                # clip from the GEMM epilogue's sums
    # the dense weights hold exactly what the masters round to
    for m in model.modules():
        if isinstance(m, M.LinearLayer_ChannelSparsity):
            master = opt.state[m.selected_weight]["master"]
            assert torch.equal(m.weight.detach()[:, m.index_list].t(), master.bfloat16())
    M.unfuse_qkv_projections(model)


def test_two_identical_native_runs_are_bit_identical(M):
    a = _train(M, True, SEL_MLP, SEL_ATTN, steps=2)
    b = _train(M, True, SEL_MLP, SEL_ATTN, steps=2)
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


# ---- one arena of channel modules of several widths ---------------------------------------------------------------

SHAPES = [(1024, 512, 77), (512, 256, 5), (256, 512, 130), (768, 256, 64)]     # (out_features, in_features, n)


def _bank(M, seed=0):
    torch.manual_seed(seed)
    layers = []
    for i, (out_f, in_f, n) in enumerate(SHAPES):
        w = torch.nn.Parameter(torch.randn(out_f, in_f, device="cuda").bfloat16() * 0.05)
        layers.append(M.LinearLayer_ChannelSparsity(w, index_list=_channels(n, in_f, 10 + i)))
    return layers


def _padded(opt, k):
    arena = opt._arenas[0]
    off, size = arena.offsets[k], arena.sizes[k]
    return arena, off, size


def test_gradients_sums_of_squares_regions_and_the_column_step(M, grouped):
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200.optim import SMTAdam
    layers = _bank(M)
    opt = SMTAdam([m.selected_weight for m in layers], lr=1e-3, betas=(0.9, 0.95), max_grad_norm=1.0)
    arena = opt._arenas[0]
    assert arena.all_sinks
    # sentinels: the padding rows of every parameter's region in the state the step must not touch, and in flat_grad
    # (where the gradient launch stores zeros)
    sentinel = {}
    for k, m in enumerate(layers):
        _a, off, size = _padded(opt, k)
        n_el = m.selected_weight.numel()
        assert size > n_el or len(m.index_list) % 64 == 0
        for name in ("master", "exp_avg", "exp_avg_sq", "flat_param", "flat_grad"):
            getattr(arena, name)[off + n_el:off + size].fill_(7.0)
        sentinel[k] = (off + n_el, off + size)
    xs = [torch.randn(3, 100, m.weight.shape[1], device="cuda").bfloat16() for m in layers]
    dys = [torch.randn(3, 100, m.weight.shape[0], device="cuda").bfloat16() for m in layers]
    w_before = [m.weight.detach().clone() for m in layers]
    opt.zero_grad()
    for m, x, dy in zip(layers, xs, dys):
        m(x).backward(dy)
    assert ops.LAST_GROUP["emits_sq"]
    for k, (m, x, dy) in enumerate(zip(layers, xs, dys)):
        truth = x.reshape(-1, x.shape[-1])[:, m.index_list].double().t() @ dy.reshape(-1, dy.shape[-1]).double()
        g = m.selected_weight.grad
        assert g.data_ptr() == arena.flat_grad[arena.offsets[k]:].data_ptr()
        assert (g.double() - truth).abs().max().item() <= 2 ** -7 * truth.abs().max().item()
        lo, hi = sentinel[k]
        assert not arena.flat_grad[lo:hi].any()                                  # rows past n: zeros
        # per-tile sums of squares of the stored values (slots [2 i, 2 i + 1] = [total, 0])
        b, rows, cols = m._grad_tiles()
        stored = arena.flat_grad[arena.offsets[k]:arena.offsets[k] + rows * b * m.weight.shape[0]]
        tiles = stored.double().view(rows, b, cols, b).pow(2).sum(dim=(1, 3)).reshape(-1)
        slot0 = m.selected_weight._smt_sink.sq_slot0
        got = arena.block_sq[slot0:slot0 + 2 * rows * cols].double().view(-1, 2)
        assert torch.allclose(got[:, 0], tiles, rtol=1e-5, atol=0) and not got[:, 1].any()
    opt.step()
    assert opt.sqnorm_source == "partials"
    for k, m in enumerate(layers):
        lo, hi = sentinel[k]
        for name in ("master", "exp_avg", "exp_avg_sq", "flat_param"):
            assert torch.equal(getattr(arena, name)[lo:hi], torch.full((hi - lo,), 7.0, device="cuda",
                                                                        dtype=getattr(arena, name).dtype)), name
        master = opt.state[m.selected_weight]["master"]
        w = m.weight.detach()
        assert torch.equal(w[:, m.index_list].t(), master.bfloat16())           # round-to-nearest-even of the master
        keep = [c for c in range(w.shape[1]) if c not in set(m.index_list)]
        assert torch.equal(w[:, keep], w_before[k][:, keep])                     # nothing else in W moved


@pytest.mark.parametrize("clip", [0.0, 1e-3])
def test_compact_adam_columns_against_the_oracle_and_the_block_kernel(M, clip):
    """Masters and moments bit-exact against oracle.adamw_fused_step and bit-identical to smt_compact_adam on the same
    slice; the selected columns are the masters rounded to bf16; every other weight element is untouched."""
    from sparse_matrix_tuning_b200 import ops
    gen = torch.Generator().manual_seed(5)
    shapes = [(256, 96, [3, 95, 40]), (1024, 64, [0, 17]), (64, 512, [511, 1, 300, 2, 8])]
    entries, total = [], 0
    for out_f, in_f, cols in shapes:
        w = (torch.randn(out_f, in_f, generator=gen) * 0.1).bfloat16().cuda()
        for c in cols:
            entries.append((w, c, total))
            total += out_f
        total += 8                                              # a gap no entry covers
    hp = dict(lr=1e-3, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.01)
    p = (torch.randn(total, generator=gen) * 0.1).float()
    m = (torch.randn(total, generator=gen) * 1e-3).float()
    v = (torch.rand(total, generator=gen) * 1e-5).float()
    g = (torch.randn(total, generator=gen) * 0.2).bfloat16()
    weights = {id(w): w for w, _c, _o in entries}
    before = {k: w.clone() for k, w in weights.items()}
    sq = (g.float() ** 2).sum().reshape(1).cuda()
    table = ops.make_column_table(entries, "cuda")
    state = [t.clone().cuda() for t in (p, m, v)]
    comp = torch.zeros(total, dtype=torch.bfloat16, device="cuda")
    ops.compact_adam(*state, g.cuda(), step=3, grad_scale=0.5, sqnorm=sq if clip else None, max_norm=clip,
                     compact_out=comp, columns=table, n_columns=len(entries), w_dtype=torch.bfloat16, **hp)
    ref = [t.clone().cuda() for t in (p, m, v)]
    ops.compact_adam(*ref, g.cuda(), step=3, grad_scale=0.5, sqnorm=sq if clip else None, max_norm=clip, **hp)
    gscale = O.clip_coef(np.float32(sq.item()), np.float32(0.5), np.float32(clip)) if clip else 0.5
    op, om, ov = O.adamw_fused_step(p.numpy(), m.numpy(), v.numpy(), g.float().numpy(), step=3, gscale=gscale, **hp)
    covered = torch.zeros(total, dtype=torch.bool)
    for w, c, off in entries:
        covered[off:off + w.shape[0]] = True
    for got, blk, want, orig in zip(state, ref, (op, om, ov), (p, m, v)):
        got = got.cpu()
        assert torch.equal(got[covered], blk.cpu()[covered])
        assert np.array_equal(got[covered].numpy().view(np.uint32), want[covered.numpy()].view(np.uint32))
        assert torch.equal(got[~covered], orig[~covered])                     # the gaps are not touched
    for w, c, off in entries:
        assert torch.equal(w[:, c].cpu(), state[0][off:off + w.shape[0]].cpu().bfloat16())
        assert torch.equal(comp[off:off + w.shape[0]], w[:, c])
    for k, w in weights.items():
        cols = {c for ww, c, _o in entries if ww is w}
        keep = [c for c in range(w.shape[1]) if c not in cols]
        assert torch.equal(w[:, keep], before[k][:, keep])


# ---- the gradient protocol, channel versions of the block tests ------------------------------------------------------

def test_no_delivery_accumulation_and_dropped_grads(M, grouped):
    from sparse_matrix_tuning_b200.optim import SMTAdam
    layer = _bank(M, seed=2)[0]
    opt = SMTAdam([layer.selected_weight], lr=1e-3)
    x = [torch.randn(2, 64, 512, device="cuda").bfloat16() for _ in range(2)]
    dy = [torch.randn(2, 64, 1024, device="cuda").bfloat16() for _ in range(2)]

    def truth(i):
        return x[i].reshape(-1, 512)[:, layer.index_list].float().t() @ dy[i].reshape(-1, 1024).float()

    opt.zero_grad()
    for i in range(2):                                      # two micro-batches accumulate
        layer(x[i]).backward(dy[i])
    want = truth(0) + truth(1)
    assert (layer.selected_weight.grad.float() - want).abs().max().item() <= 2 ** -6 * want.abs().max().item()
    opt.step()
    layer.selected_weight.grad = None                       # model.zero_grad(set_to_none=True)
    layer(x[0]).backward(dy[0])
    assert layer.selected_weight.grad.data_ptr() == opt.flat_grads()[0].data_ptr()
    want = truth(0)
    assert (layer.selected_weight.grad.float() - want).abs().max().item() <= 2 ** -7 * want.abs().max().item()
    opt.step()
    m_before = opt.state[layer.selected_weight]["exp_avg"].clone()
    opt.zero_grad()
    opt.step()                                              # no delivery after zero_grad: the step sees zeros
    assert not opt.flat_grads()[0].any()
    assert torch.allclose(opt.state[layer.selected_weight]["exp_avg"], m_before * 0.9)


def test_forward_skips_the_scatter_only_while_smtadam_vouches(M):
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200.optim import SMTAdam
    layer = _bank(M, seed=3)[1]
    opt = SMTAdam([layer.selected_weight], lr=1e-2)
    x = torch.randn(2, 16, 256, device="cuda").bfloat16()

    def columns_match():
        return torch.equal(layer.weight.detach()[:, layer.index_list].t(), layer.selected_weight.detach())

    opt.zero_grad()
    layer(x).float().pow(2).mean().backward()
    opt.step()
    assert columns_match()
    n0 = ops.LAUNCHES["total"]
    with torch.no_grad():
        layer(x)
    assert ops.LAUNCHES["total"] == n0 + 1                  # the channel gather only: no scatter
    with torch.no_grad():
        layer.selected_weight.add_(0.5)                     # a version-counted write: the forward scatters again
        layer(x)
    assert ops.LAUNCHES["total"] == n0 + 3
    assert columns_match()
    opt.zero_grad()
    layer(x).float().pow(2).mean().backward()
    opt.step()
    layer.selected_weight.data = layer.selected_weight.data.clone() * 3     # re-pointed storage: no longer vouched for
    n1 = ops.LAUNCHES["total"]
    with torch.no_grad():
        layer(x)
    assert ops.LAUNCHES["total"] == n1 + 2
    assert columns_match()


def test_deepcopy_export_and_overlapped_exchange(M):
    from sparse_matrix_tuning_b200 import checkpoint as CK, dp
    from sparse_matrix_tuning_b200.optim import SMTAdam
    model = _model(M, SEL_MLP, SEL_ATTN, fuse=True)
    twin = copy.deepcopy(model)
    ids = torch.randint(0, 512, (2, 64), generator=torch.Generator().manual_seed(4)).cuda()
    with torch.no_grad():
        before = twin(input_ids=ids, use_cache=False).logits
        for n, p in model.named_parameters():
            if any(k in n for k in ("q_proj", "k_proj", "v_proj", "norm")):
                p.mul_(-3.0)
        after = twin(input_ids=ids, use_cache=False).logits
    assert torch.equal(before, after)
    layer = twin.model.layers[0]
    assert layer.self_attn.q_proj._smt_shared_group.members[0] is layer.self_attn.q_proj

    # single-GPU overlapped exchange with channel sinks == the plain all-reduce path
    def run(overlap):
        m = _model(M, SEL_MLP, SEL_ATTN, fuse=True)
        opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(m, 0.0, 1e-3), betas=(0.9, 0.95), max_grad_norm=1.0)
        M.set_grouped_backward(True, chunk_blocks=8 if overlap else 0)
        ex = dp.OverlappedGradExchange(opt, sqnorm=True) if overlap else None
        try:
            opt.zero_grad()
            m(input_ids=ids, labels=ids, use_cache=False).loss.backward()
            if ex is not None:
                # every channel gradient went through a grouped flush and its listener, chunk by chunk
                assert len(ex.reduced_ranges) >= 2
                assert sum(n for _o, n in ex.reduced_ranges) == sum(sk.view.numel() for sk in opt._arenas[0].sinks)
                ex.finish()
                assert opt._arenas[0].sq_override is not None
            else:
                dp.allreduce_compact_grads(opt)
            grads = opt.flat_grads()[0].clone()
            opt.step()
            return grads, m, opt
        finally:
            if ex is not None:
                ex.close()
            M.set_grouped_backward(False)

    g0, _m0, _o0 = run(False)
    g1, m1, o1 = run(True)
    assert torch.equal(g0, g1)
    assert o1.sqnorm_source == "partials"
    # the merged export after native steps carries the trained columns
    merged = CK.merged_state_dict(m1)
    q = m1.model.layers[0].self_attn.q_proj
    w = merged["model.layers.0.self_attn.q_proj.weight"]
    assert torch.equal(w[:, q.index_list].t(), o1.state[q.selected_weight]["master"].bfloat16())
    assert not any("selected_weight" in k for k in merged)
    M.unfuse_qkv_projections(m1)
    M.convert_channel_sparsity_to_linear_layer(m1)
    assert not any(isinstance(x, M.LinearLayer_ChannelSparsity) for x in m1.modules())
    assert torch.equal(m1.model.layers[0].self_attn.q_proj.weight, w)
