"""GPU tests of the factored warm-up block sums: `smt_token_block_sums` and `smt_block_outer_accumulate` against fp64,
and `FactoredBlockSumAccumulator` on small LLaMA models - against the fp64 truth recorded from the same pass and
against the existing bf16-gradient path, selection parity with BASELINE config 1, checkpointing modes, the fused frozen
model and the unfuse -> convert -> fuse flow after warm-up."""
import copy

import pytest
import torch

from conftest import load_golden
from oracle import golden_inputs as GI
from oracle import smt_oracle as O

pytestmark = pytest.mark.gpu

KINDS_ATTN = ("q_proj", "k_proj", "v_proj")
KINDS_MLP = ("gate_proj", "up_proj", "down_proj")


@pytest.fixture(scope="module")
def lib(built_library):
    return built_library


def _segment_truth(x, b):
    T, F = x.shape
    xd = x.double().reshape(T, F // b, b)
    return xd.sum(-1), xd.abs().sum(-1)


# ---- 1. token_block_sums ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("F", [1024, 4096, 14336])
def test_token_block_sums_against_fp64(lib, dtype, F):
    from sparse_matrix_tuning_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(F)
    T = 333
    wide = (torch.randn(T, F + 64, device="cuda", generator=g) * 3 + 0.5).to(dtype)
    for x in (wide[:, :F].contiguous(), wide[:, :F], wide[:, 64:]):          # contiguous, and row pitch F + 64
        for b in (64, 128, 256):
            got = ops.token_block_sums(x, b)
            assert got.shape == (T, F // b) and got.dtype == torch.float32
            truth, bound = _segment_truth(x, b)
            assert ((got.double() - truth).abs() <= 1e-5 * bound).all(), (b, x.stride())
            assert torch.equal(got, ops.token_block_sums(x, b))                 # bit-identical across calls


def test_token_block_sums_token_counts(lib):
    from sparse_matrix_tuning_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(8191, 4096 + 128, device="cuda", generator=g).bfloat16()[:, :4096]
    for b in (64, 128, 256):
        full = ops.token_block_sums(x, b)
        truth, bound = _segment_truth(x, b)
        assert ((full.double() - truth).abs() <= 1e-5 * bound).all()
        one = ops.token_block_sums(x[:1], b)
        assert torch.equal(one, full[:1])          # a segment's bits do not depend on T or on the grid
        assert torch.equal(ops.token_block_sums(x[4000:4077], b), full[4000:4077])
        empty = ops.token_block_sums(x[:0], b)
        assert empty.shape == (0, 4096 // b)


# ---- 2. block_outer_accumulate -------------------------------------------------------------------------------------

@pytest.mark.parametrize("rb,cb", [(16, 16), (16, 56), (56, 16), (224, 64), (3, 5)])
def test_block_outer_accumulate_against_fp64(lib, rb, cb):
    from sparse_matrix_tuning_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(rb * 1000 + cb)
    for T in (1, 127, 129, 511, 512, 513, 1000, 8192):
        dy = torch.randn(T, rb, device="cuda", generator=g) * 5
        x = torch.randn(T, cb, device="cuda", generator=g) * 7
        start = torch.randn(rb, cb, device="cuda", generator=g)
        got = start.clone()
        ops.block_outer_accumulate(got, dy, x)
        truth = start.double() + dy.double().t() @ x.double()
        bound = dy.double().abs().t() @ x.double().abs() + start.double().abs()
        assert ((got.double() - truth).abs() <= 1e-5 * bound).all(), T
        again = start.clone()
        ops.block_outer_accumulate(again, dy, x)
        assert torch.equal(again, got), T                                     # bit-identical across calls
    ops.block_outer_accumulate(got, dy[:0], x[:0])                          # T = 0: nothing changes
    assert torch.equal(again, got)


# ---- model helpers ---------------------------------------------------------------------------------------------------

def _model(layers=2, seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=512, hidden_size=512, intermediate_size=1024, num_hidden_layers=layers,
                      num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=256,
                      attn_implementation="sdpa")
    torch.manual_seed(seed)
    model = LlamaForCausalLM(cfg).cuda().bfloat16()
    model.config.use_cache = False
    return model


def _freeze(model):
    for p in model.parameters():
        p.requires_grad_(False)
    model.enable_input_require_grads()
    return model


def _ids(n, seed=1, B=2, S=128):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 512, (B, S), generator=g).cuda() for _ in range(n)]


def _math_attention():
    from torch.nn.attention import SDPBackend, sdpa_kernel
    return sdpa_kernel(SDPBackend.MATH)


class _Recorder:
    """Keeps x and dy of every targeted Linear of one pass (fp64) and forms the exact block sums from them."""

    def __init__(self, model, mlp):
        from sparse_matrix_tuning_b200.warmup import classify_parameter
        self.x, self.dy, self.handles = {}, {}, []
        for name, mod in model.named_modules():
            key = classify_parameter(name + ".weight", mlp, True) if isinstance(mod, torch.nn.Linear) else None
            if key is not None:
                self.handles.append(mod.register_forward_hook(lambda _m, a, o, key=key: self._fwd(key, a[0], o)))

    def _fwd(self, key, x, out):
        if not out.requires_grad:
            return
        assert key not in self.x
        self.x[key] = x.detach().reshape(-1, x.shape[-1]).double()
        out.register_hook(lambda g: self.dy.__setitem__(key, g.detach().reshape(-1, g.shape[-1]).double()))

    def remove(self):
        for h in self.handles:
            h.remove()

    def truth(self, b):
        """{key: (fp64 block sums, sum of |terms| per block)}"""
        out = {}
        for key, x in self.x.items():
            dy = self.dy[key]
            T = x.shape[0]
            X, Xa = x.view(T, -1, b).sum(-1), x.abs().view(T, -1, b).sum(-1)
            D, Da = dy.view(T, -1, b).sum(-1), dy.abs().view(T, -1, b).sum(-1)
            out[key] = (D.t() @ X, Da.t() @ Xa)
        return out


def _within(acc, truth, rel=1e-5):
    assert set(acc) == set(truth)
    for key, (t, bound) in truth.items():
        err = (acc[key].double() - t).abs()
        assert (err <= rel * bound).all(), (key, (err / bound).max().item())


def _pass(model, ids):
    model(input_ids=ids, labels=ids, use_cache=False).loss.backward()


# ---- 3. same pass, two accumulators ----------------------------------------------------------------------------------

def test_same_pass_against_truth_and_the_bf16_gradient_path(lib):
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator, WarmupGradAccumulator
    model = _model()
    for n, p in model.named_parameters():
        p.requires_grad_(any(k in n for k in KINDS_ATTN + KINDS_MLP))
    model.train()
    new = FactoredBlockSumAccumulator(block=256, mlp=True).attach(model)
    old = WarmupGradAccumulator(block=256, mode="block_sum", mlp=True)
    old.attach(model, free_grads=True)
    rec = _Recorder(model, mlp=True)
    with _math_attention():
        _pass(model, _ids(1)[0])
    torch.cuda.synchronize()
    new.detach()
    old.detach()
    rec.remove()
    assert {k for k, _l in new.acc} == set(KINDS_ATTN + KINDS_MLP) and len(new.acc) == 12
    assert set(new.acc) == set(old.acc) and all(new.shapes[k] == old.shapes[k] for k in new.acc)
    truth = rec.truth(256)
    _within(new.acc, truth)
    for key, (t, _bound) in truth.items():
        err_new = (new.acc[key].double() - t).abs().max().item()
        err_old = (old.acc[key].double() - t).abs().max().item()
        assert err_new <= err_old, (key, err_new, err_old)
    keys, scores = new.scores("mean_abs")
    assert keys == list(new.acc)
    assert all(torch.equal(s, (new.acc[k] / 65536).abs()) for k, s in zip(keys, scores))


# ---- 4. reference parity ---------------------------------------------------------------------------------------------

def test_config1_selection_from_factored_sums(lib):
    """BASELINE config 1 (fp32), frozen weights: the factored warm-up selects exactly what the reference selected from
    its accumulated weight gradients."""
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    gold = load_golden("config1_e2e.pt")
    c = GI.CONFIG1
    model, batches = GI.make_config1(device="cuda")
    named = list(model.named_parameters())
    n_attn = O.block_budget(named, c["attn_ratio"])
    assert n_attn == gold["n_attn"]
    _freeze(model)
    acc = FactoredBlockSumAccumulator(block=256).attach(model)
    for it in range(c["warmup_steps"]):
        out = model(input_ids=batches[it], labels=batches[it], use_cache=False)
        out.loss.backward()
        assert abs(out.loss.item() - gold["warm_losses"][it]) <= 5e-5
    acc.detach()
    keys, scores = acc.scores("mean_abs")
    sel = H.select_submatrix_from_scores(keys, scores, n_attn, "no_restriction")
    flat = torch.cat([s.reshape(-1) for s in scores]).sort(descending=True).values
    gap = (flat[n_attn - 1] - flat[n_attn]).item() / flat[n_attn - 1].item()
    print(f"config 1: relative score gap at the cut-off {gap:.3e}")
    assert [(k, list(v)) for k, v in sel.items()] == [(k, [tuple(t) for t in v]) for k, v in gold["selection"]], \
        f"relative gap at the cut-off: {gap:.3e}"


# ---- 5. checkpointing modes --------------------------------------------------------------------------------------------

def test_checkpointing_modes_agree(lib):
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    model = _freeze(_model())
    model.train()
    ids = _ids(1)[0]

    def run(mode, record=False):
        model.gradient_checkpointing_disable()
        if mode is not None:
            model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": mode == "reentrant"})
        acc = FactoredBlockSumAccumulator(block=256, mlp=True).attach(model)
        rec = _Recorder(model, mlp=True) if record else None
        with _math_attention():
            _pass(model, ids)
        torch.cuda.synchronize()
        acc.detach()
        if rec is not None:
            rec.remove()
        return acc.acc, rec

    base, rec = run(None, record=True)
    truth = rec.truth(256)
    for mode in (None, "non_reentrant", "reentrant"):
        a = run(mode)[0]
        b = run(mode)[0]
        assert all(torch.equal(a[k], b[k]) for k in a), mode                 # bit-identical within a mode
        _within(a, truth)                                                     # kernel tolerance across modes
    model.gradient_checkpointing_disable()


# ---- 6. fused, frozen model ---------------------------------------------------------------------------------------------

def test_fused_frozen_model_and_the_flow_after_warm_up(lib):
    from sparse_matrix_tuning_b200.optim import SMTAdam
    from sparse_matrix_tuning_b200.smt import smt as M, smt_helper as H
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    plain = _freeze(_model(layers=3))
    fused = copy.deepcopy(plain)
    assert M.fuse_qkv_projections(fused) == 3 and M.fuse_causal_lm_loss(fused)
    batches = _ids(4, seed=5)

    def warm(model):
        acc = FactoredBlockSumAccumulator(block=256, mlp=True).attach(model)
        with _math_attention():
            for ids in batches[:2]:
                _pass(model, ids)
        torch.cuda.synchronize()
        acc.detach()
        return acc

    acc_p, acc_f = warm(plain), warm(fused)
    assert list(acc_f.acc) == list(acc_p.acc) and len(acc_f.acc) == 18
    worst = 0.0
    for key in acc_f.acc:
        assert acc_f.acc[key].abs().sum() > 0, key                            # every targeted module contributes
        rel = ((acc_f.acc[key] - acc_p.acc[key]).norm() / acc_p.acc[key].norm()).item()
        # the fused path rounds differently (tcgen05 GEMMs, native norms, chunked loss), so dy differs at bf16 level
        assert rel <= 5e-2, (key, rel)
        worst = max(worst, rel)
    print(f"fused vs unfused frozen model, relative L2 of the block sums: max {worst:.3e}")

    keys, scores = acc_p.scores("mean_abs")
    sel = H.select_submatrix_from_scores(keys, scores, 12, "no_restriction")
    sel_attn = {k: v for k, v in sel.items() if k[0] in KINDS_ATTN}
    sel_mlp = {k: v for k, v in sel.items() if k[0] in KINDS_MLP}

    def train(model):
        M.freeze_unselected_matrix_layer(model, sel_mlp, sel_attn)
        M.convert_linear_layer_to_matrix_sparsity(model, sel_mlp, sel_attn)
        M.fuse_qkv_projections(model)
        M.fuse_causal_lm_loss(model)
        opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-3), betas=(0.9, 0.95),
                      max_grad_norm=1.0)
        out = []
        for ids in batches[2:]:
            opt.zero_grad()
            loss = model(input_ids=ids, labels=ids, use_cache=False).loss
            loss.backward()
            out.append((loss.detach().clone(), [g.clone() for g in opt.flat_grads()]))
            opt.step()
        return out

    assert M.unfuse_qkv_projections(fused) == 3
    got, want = train(fused), train(plain)
    for (l1, g1), (l2, g2) in zip(got, want):
        assert torch.equal(l1, l2)
        assert len(g1) == len(g2) and all(torch.equal(a, b) for a, b in zip(g1, g2))


# ---- 7. other behaviour -----------------------------------------------------------------------------------------------

def test_gradient_accumulation_and_no_grad_forwards(lib):
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    model = _freeze(_model())
    model.train()
    b1, b2 = _ids(2, seed=7)

    def run(batches, no_grad_between=False):
        acc = FactoredBlockSumAccumulator(block=256, mlp=True).attach(model)
        with _math_attention():
            for i, ids in enumerate(batches):
                _pass(model, ids)
                if no_grad_between and i == 0:
                    torch.cuda.synchronize()
                    snap = {k: v.clone() for k, v in acc.acc.items()}
                    with torch.no_grad():
                        model(input_ids=ids, use_cache=False)
                    torch.cuda.synchronize()
                    assert all(torch.equal(snap[k], acc.acc[k]) for k in snap)
        torch.cuda.synchronize()
        acc.detach()
        return acc.acc

    one, two = run([b1]), run([b2])
    both = run([b1, b2], no_grad_between=True)
    assert {k for k, _l in both} == set(KINDS_ATTN + KINDS_MLP)
    for k in both:
        assert torch.equal(both[k], one[k] + two[k]), k        # the second pass adds its (fp32) sum onto the first
