"""CPU tests that PIN the oracle (oracle/smt_oracle.py): against the committed golden vectors produced by the
unmodified reference (oracle/gen_golden.py), and against the live reference whenever /root/reference exists."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import golden_inputs as GI
from oracle import smt_oracle as O
from oracle.ref_shim import load_reference, reference_available


def _as_dict(pairs):
    return {k: list(map(tuple, v)) for k, v in pairs}


@pytest.mark.parametrize("case", load_golden("selection_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_selection_matches_reference_golden(case):
    spec = case["spec"]
    grads, dims = GI.make_selection_inputs(spec)
    assert GI.tensor_dict_sha(grads) == case["input_sha"], "seeded inputs drifted from the ones the golden was made with"
    if "raises" in case:
        assert case["raises"] == "UnboundLocalError"      # the reference dies at smt_helper.py:142 for n == 0
        with pytest.raises(UnboundLocalError):
            O.select_submatrix(grads, dims, spec["n"], spec["selection_strategy"], spec["calculate_strategy"])
        return
    got = O.select_submatrix(grads, dims, spec["n"], spec["selection_strategy"], spec["calculate_strategy"])
    assert list(got.keys()) == [k for k, _ in case["selection"]]          # dict insertion order too
    assert _as_dict(got.items()) == _as_dict(case["selection"])
    for key, ref_scores in case["scores"].items():
        mine = O.block_scores(grads[key], 256, spec["calculate_strategy"], dims[key[0]])
        assert torch.equal(mine, ref_scores)


@pytest.mark.parametrize("case", load_golden("channel_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_channel_selection_matches_reference_golden(case):
    spec = case["spec"]
    act = GI.make_channel_inputs(spec)
    assert GI.tensor_dict_sha(act) == case["input_sha"]
    got = O.select_channels(act, spec["n"], spec["selection_strategy"], spec["calculate_strategy"])
    assert {k: list(v) for k, v in got.items()} == {k: list(v) for k, v in case["selection"]}


@pytest.mark.parametrize("case", load_golden("linearz_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_linearz_matches_reference_golden(case):
    spec, b = case["spec"], case["spec"]["block"]
    x, dy, w, idx = case["x"], case["dy"], case["w"], case["index_list"]
    sel0 = O.gather_blocks(w, idx, b)
    assert torch.equal(sel0, case["selected0"])
    w2 = O.scatter_blocks(w.clone(), sel0 * 0.5, idx, b)
    assert GI.tensor_dict_sha({"w": w2}) == case["w_after_sha"]
    assert torch.equal(O.linearz_forward(x, w2), case["y"])
    gi, gw = O.linearz_backward(x, dy, w2, idx, b)
    assert torch.equal(gw, case["grad_weight"])
    assert torch.equal(gi, case["grad_input"])


@pytest.mark.parametrize("case", load_golden("linearchannel_cases.pt"), ids=lambda c: c["spec"]["name"])
def test_linearchannel_matches_reference_golden(case):
    """The reference's channel layer on square weights (the only shapes it runs on): same y, grad_input and [n, out]
    channel gradient, bit for bit.  The column gather / scatter restatement round-trips."""
    x, dy, w, idx = case["x"], case["dy"], case["w"], case["index_list"]
    assert torch.equal(O.linearz_forward(x, w), case["y"])
    gi, gw = O.linearchannel_backward(x, dy, w, idx)
    assert torch.equal(gw, case["grad_weight"]) and torch.equal(gi, case["grad_input"])
    cols = O.gather_columns(w, idx)
    assert cols.shape == (len(idx), w.shape[0]) and torch.equal(cols[0], w[:, idx[0]])
    w2 = O.scatter_columns(w.clone(), cols * 2, idx)
    keep = [c for c in range(w.shape[1]) if c not in idx]
    assert torch.equal(w2[:, idx], w[:, idx] * 2) and torch.equal(w2[:, keep], w[:, keep])


def test_config1_budget_and_dims_match_golden():
    gold = load_golden("config1_e2e.pt")
    model, _ = GI.make_config1()
    named = list(model.named_parameters())
    assert O.targeted_module_dims(named) == gold["dims"]
    assert O.block_budget(named, GI.CONFIG1["attn_ratio"]) == gold["n_attn"] == 5
    assert gold["total_blocks"] == 596


@pytest.mark.skipif(not reference_available(), reason="the original project's smt modules are not staged (oracle/build_ref.py)")
def test_oracle_against_live_reference():
    S, H = load_reference()
    torch.manual_seed(5)
    grads = {("q_proj", 0): torch.randn(512, 768), ("k_proj", 0): torch.randn(256, 768),
             ("v_proj", 0): torch.randn(256, 768), ("q_proj", 1): torch.randn(512, 768)}
    dims = {"q_proj": [512, 768], "k_proj": [256, 768], "v_proj": [256, 768]}
    for cs in ("mean_abs", "abs_mean", "L1", "L2"):
        for ss in ("no_restriction", "norm_dist"):
            ref = H.select_submatrix_based_on_grads(grads, dims, 4, selection_strategy=ss, calculate_strategy=cs)
            mine = O.select_submatrix(grads, dims, 4, ss, cs)
            assert list(ref.items()) == list(mine.items())
    # linearZ, bf16, patched block size
    x = torch.randn(3, 20, 256).bfloat16(); dy = torch.randn(3, 20, 128).bfloat16()
    w = (torch.randn(128, 256) * 0.02).bfloat16(); idx = [(1, 2), (0, 0), (1, 3)]
    S.Block_dimension = 64
    try:
        layer = S.LinearLayer_MatrixSparsity(torch.nn.Parameter(w.clone()), index_list=idx)
        xin = x.clone().requires_grad_(True)
        y = layer(xin); y.backward(dy)
    finally:
        S.Block_dimension = 256
    gi, gw = O.linearz_backward(x, dy, w, idx, 64)
    assert torch.equal(gw, layer.selected_weight.grad) and torch.equal(gi, xin.grad)
    assert torch.equal(O.linearz_forward(x, w), y)


def test_adam_restatement_agrees_with_torch_adamw():
    """Parity UNPINNED against DeepSpeed (not vendored); the restated update must at least agree with
    torch.optim.AdamW in fp32 to 1e-6 relative over several steps."""
    rng = np.random.RandomState(0)
    p = rng.randn(4096).astype(np.float32); m = np.zeros_like(p); v = np.zeros_like(p)
    tp = torch.nn.Parameter(torch.from_numpy(p.copy()))
    opt = torch.optim.AdamW([tp], lr=1e-3, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.01)
    for step in range(1, 6):
        g = (rng.randn(4096) * 0.1).astype(np.float32)
        p, m, v = O.adamw_fused_step(p, m, v, g, lr=1e-3, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.01, step=step)
        tp.grad = torch.from_numpy(g.copy()); opt.step()
        assert np.max(np.abs(p - tp.detach().numpy())) <= 1e-6 * max(1.0, np.abs(p).max())


def test_clip_coef_matches_torch_clip_grad_norm():
    g = torch.randn(1000) * 3
    sq = np.float32((g.double() ** 2).sum().item())
    scale = O.clip_coef(sq, np.float32(1.0), np.float32(1.0))
    t = g.clone().requires_grad_(True); t.grad = g.clone()
    torch.nn.utils.clip_grad_norm_([t], 1.0)
    assert torch.allclose(t.grad, g * float(scale), rtol=1e-6, atol=0)
    assert O.clip_coef(np.float32(0.01), np.float32(1.0), np.float32(1.0)) == np.float32(1.0)


def test_bf16_round_matches_torch():
    a = torch.randn(10000) * 100
    assert np.array_equal(O.bf16_round(a.numpy()), a.bfloat16().float().numpy())
