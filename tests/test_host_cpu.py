"""CPU tests of the host side: the C-ABI library loads and exports every symbol the header declares, argument
validation works without a GPU, the host logic (tuple-order ranks, parameter classification, freezing,
parameter groups) mirrors the reference, and the product path fails LOUDLY without CUDA (no CPU fallback)."""
import ctypes
import os
import re
import warnings

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import golden_inputs as GI
from oracle import smt_oracle as O
from oracle.ref_shim import load_reference, reference_available

NOT_STAGED = "the original project's smt modules are not staged (oracle/build_ref.py): comparison with them not run"


def test_library_exports_every_header_symbol(built_library):
    header = open(os.path.join(ROOT, "include", "smt_b200.h")).read()
    declared = set(re.findall(r"\b(smt_[a-z0-9_]+)\s*\(", header))
    declared -= {"smt_block_ref"}
    assert len(declared) >= 19
    from sparse_matrix_tuning_b200 import _lib
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), f"{name} declared in include/smt_b200.h but not exported"
    assert built_library.smt_version() >= 200


def test_block_ref_struct_layout():
    from sparse_matrix_tuning_b200._lib import BlockRef
    assert ctypes.sizeof(BlockRef) == 24
    assert BlockRef.ldw.offset == 8 and BlockRef.row.offset == 16 and BlockRef.col.offset == 20


def test_argument_validation_needs_no_gpu(built_library):
    lib = built_library
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p).value
    assert lib.smt_block_score_reduce(p, 512, 512, 512, 100, 0, p, None) == -1
    assert b"block size 100" in lib.smt_last_error()
    assert lib.smt_block_score_reduce(p, 500, 512, 512, 256, 0, p, None) == -1
    assert lib.smt_block_score_reduce(p, 512, 512, 512, 256, 9, p, None) == -1
    assert b"strategy" in lib.smt_last_error()
    assert lib.smt_score_accumulate(None, None, 1, 8, None) == -1
    assert lib.smt_block_grad_gemm(p, 512, 500, p, 512, 512, 64, 1, p, 1, 256, p, 1, 0, None, 0, None) == -1
    assert b"multiples of block" in lib.smt_last_error()
    assert lib.smt_block_grad_gemm_run_width(256) == 0                                   # b = 256 has no run tiles
    assert lib.smt_block_grad_gemm_runs(p, 512, 512, p, 512, 512, 64, 1, p, 1, 256, p, 1, 0, None, 0, None) == -1
    assert b"block size 256" in lib.smt_last_error()
    assert lib.smt_compact_adam(p, p, p, p, 1, 12, 1e-3, .9, .95, 1e-8, 0., .1, .05, 1., None, 0, 0., None, 1, None, 0, 0, 1, None) == -1
    assert lib.smt_topk_blocks(p, p, None, 8, p, p, p, 1, p, p, 1 << 20, None) == -1      # rank without inverse
    assert lib.smt_topk_workspace_bytes(1000) >= 16000
    assert lib.smt_block_grad_gemm_workspace_bytes(0, 256, 1024, 1) == 0
    # zero-sized work is a no-op that needs no device
    assert lib.smt_block_grad_gemm(None, 0, 512, None, 0, 512, 0, 1, None, 0, 256, None, 1, 0, None, 0, None) == 0
    assert lib.smt_block_gather(None, 0, 256, 2, None, None) == 0


def test_plan_is_deterministic_and_bounded(built_library):
    from sparse_matrix_tuning_b200 import ops
    s1 = ops.block_grad_gemm_plan(9, 256, 8192, torch.bfloat16)
    assert s1 == ops.block_grad_gemm_plan(9, 256, 8192, torch.bfloat16)
    splits, ctas = s1
    assert splits >= 1 and ctas in (9 * splits, 18 * splits)      # whole-block or half-block tiles
    assert splits > 1                                             # 9 blocks cannot fill 148 SMs without split-K
    assert ops.block_grad_gemm_plan(500, 256, 8192, torch.bfloat16) == (1, 500)
    assert ops.block_grad_gemm_plan(3, 64, 64, torch.bfloat16)[0] == 1
    assert ops.block_grad_gemm_plan(3, 128, 512, torch.float32) == (1, 12)


def test_tuple_order_ranks_match_python_sort():
    from sparse_matrix_tuning_b200.smt.smt_helper import _tuple_order_ranks
    keys = [("q_proj", 0), ("k_proj", 0), ("v_proj", 0), ("q_proj", 10), ("k_proj", 9), ("v_proj", 2), ("down_proj", 1)]
    shapes = [(2, 2), (1, 2), (1, 2), (2, 2), (1, 2), (1, 2), (2, 6)]
    sizes = [a * b for a, b in shapes]
    rank, inv = _tuple_order_ranks(keys, sizes)
    flat = [(k, i, j) for k, (r, c) in zip(keys, shapes) for i in range(r) for j in range(c)]
    order = sorted(range(len(flat)), key=lambda t: flat[t])
    expect = np.empty(len(flat), dtype=np.int64)
    expect[order] = np.arange(len(flat))
    assert rank.tolist() == expect.tolist()
    assert inv[rank].tolist() == list(range(len(flat)))


def test_classify_parameter_matches_capture_loop():
    from sparse_matrix_tuning_b200.warmup import classify_parameter
    model, _ = GI.make_config1()
    names = [n for n, _ in model.named_parameters()]
    got = {n: classify_parameter(n, mlp=True, attention=True) for n in names}
    fake = {n: torch.zeros(1) for n in names}
    acc = O.warmup_accumulate({}, fake.items(), mlp=True, attention=True)
    assert set(k for k in got.values() if k is not None) == set(acc.keys())
    assert got["model.layers.1.self_attn.o_proj.weight"] is None
    assert got["model.layers.0.self_attn.k_proj.weight"] == ("k_proj", 0)
    assert classify_parameter("model.layers.0.mlp.up_proj.weight", mlp=False, attention=True) is None


def _tiny_llama():
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=512, hidden_size=256, intermediate_size=512, num_hidden_layers=3,
                      num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=64)
    return LlamaForCausalLM(cfg)


@pytest.mark.parametrize("mixture,layernorm", [(False, False), (True, False), (True, True)])
def test_freeze_matches_reference(mixture, layernorm):
    from sparse_matrix_tuning_b200.smt import smt as M
    sel_mlp = {("up_proj", 1): [(0, 0)], ("down_proj", 2): [(0, 1)]}
    sel_attn = {("q_proj", 0): [(0, 0)], ("v_proj", 2): [(0, 0)], ("o_proj", 1): [(0, 0)]}
    if mixture:
        sel_mlp = {**sel_mlp, **sel_attn, ("embed_tokens", None): [(0, 0)]}
    mine = M.freeze_unselected_matrix_layer(_tiny_llama(), sel_mlp, sel_attn, mixture=mixture, layernorm=layernorm)
    flags = {n: p.requires_grad for n, p in mine.named_parameters()}
    if reference_available():
        S, _ = load_reference()
        ref = S.freeze_unselected_matrix_layer(_tiny_llama(), sel_mlp, sel_attn, mixture=mixture, layernorm=layernorm)
        assert flags == {n: p.requires_grad for n, p in ref.named_parameters()}
    else:
        warnings.warn(NOT_STAGED)
    assert flags["model.layers.1.mlp.up_proj.weight"] and not flags["model.layers.0.mlp.up_proj.weight"]
    assert not flags["lm_head.weight"] and not flags["model.norm.weight"]
    assert flags["model.layers.1.self_attn.o_proj.weight"]        # smt.py:732 dispatches o_proj too
    assert flags["model.embed_tokens.weight"] == mixture
    assert flags["model.layers.0.input_layernorm.weight"] == (mixture and layernorm)


def test_param_groups_match_reference():
    from sparse_matrix_tuning_b200.smt import smt as M
    model = _tiny_llama()
    for n, p in model.named_parameters():
        p.requires_grad = ("q_proj" in n) or ("input_layernorm" in n)
    groups = M.get_optimizer_sparse_grouped_parameters(model, 0.1, 3e-4)
    assert [len(g["params"]) for g in groups] == [3, 3]
    assert groups[0]["lr"] == 3e-4 and groups[0]["weight_decay"] == 0.1
    assert groups[1]["weight_decay"] == 0.0 and "lr" not in groups[1]
    qk = M.get_optimizer_qk_augment_grouped_parameters(model, 0.0, 1e-5, module_lr=7e-4)
    assert qk[0]["lr"] == 7e-4 and len(qk[0]["params"]) == 3       # only q_proj trainable => the "module" group
    if reference_available():
        S, _ = load_reference()
        ref = S.get_optimizer_sparse_grouped_parameters(model, 0.1, 3e-4)
        assert len(ref) == len(groups)
        for a, b in zip(ref, groups):
            assert [id(p) for p in a["params"]] == [id(p) for p in b["params"]]
            assert {k: v for k, v in a.items() if k != "params"} == {k: v for k, v in b.items() if k != "params"}
    else:
        warnings.warn(NOT_STAGED)


def test_public_api_names_and_signatures():
    import inspect
    from sparse_matrix_tuning_b200.smt import smt as M, smt_helper as H
    for name in ("convert_linear_layer_to_matrix_sparsity", "get_optimizer_sparse_grouped_parameters",
                 "get_optimizer_qk_augment_grouped_parameters", "freeze_unselected_matrix_layer",
                 "freeze_unselected_channel_layer", "convert_linear_layer_to_channel_sparsity",
                 "convert_matrix_sparsity_to_linear_layer", "LinearLayer_MatrixSparsity", "linearZ",
                 "LinearLayer_ChannelSparsity", "linearChannel"):
        assert hasattr(M, name)
    for name in ("select_submatrix_based_on_grads", "get_blocks", "get_named_linears",
                 "select_channel_based_on_activation"):
        assert hasattr(H, name)
    assert M.Block_dimension == 256
    if reference_available():
        S, RH = load_reference()
        for mod, ref, names in ((M, S, ("convert_linear_layer_to_matrix_sparsity", "freeze_unselected_matrix_layer",
                                        "get_optimizer_sparse_grouped_parameters", "convert_matrix_sparsity_to_linear_layer",
                                        "get_optimizer_qk_augment_grouped_parameters",
                                        "convert_linear_layer_to_channel_sparsity", "freeze_unselected_channel_layer")),
                                (H, RH, ("select_submatrix_based_on_grads", "select_channel_based_on_activation"))):
            for n in names:
                a, b = inspect.signature(getattr(mod, n)), inspect.signature(getattr(ref, n))
                assert list(a.parameters) == list(b.parameters), n
                assert [p.default for p in a.parameters.values()] == [p.default for p in b.parameters.values()], n
        assert list(inspect.signature(M.LinearLayer_MatrixSparsity.__init__).parameters) == \
            list(inspect.signature(S.LinearLayer_MatrixSparsity.__init__).parameters)
        assert list(inspect.signature(M.LinearLayer_ChannelSparsity.__init__).parameters) == \
            list(inspect.signature(S.LinearLayer_ChannelSparsity.__init__).parameters)
    else:
        warnings.warn(NOT_STAGED)


def test_freeze_unselected_channel_layer_matches_reference():
    """smt.py:748-831 on a tiny LLaMA: same requires_grad pattern as the reference, with and without mixture."""
    if not reference_available():
        pytest.skip("reference not mounted")
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200.smt import smt as M
    S, _ = load_reference()
    cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, vocab_size=128)
    sel_mlp = {("gate_proj", 0): [1, 2], ("down_proj", 1): [3]}
    sel_attn = {("q_proj", 1): [5], ("v_proj", 0): [0, 7], ("o_proj", 0): [1]}
    for mixture in (False, True):
        torch.manual_seed(0)
        a, b = LlamaForCausalLM(cfg), LlamaForCausalLM(cfg)
        merged = {**sel_mlp, **sel_attn}
        S.freeze_unselected_channel_layer(a, merged if mixture else sel_mlp, sel_attn, mixture=mixture)
        M.freeze_unselected_channel_layer(b, merged if mixture else sel_mlp, sel_attn, mixture=mixture)
        assert [(n, p.requires_grad) for n, p in a.named_parameters()] == \
            [(n, p.requires_grad) for n, p in b.named_parameters()]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour WITHOUT a GPU")
def test_product_path_fails_loudly_without_cuda():
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    from sparse_matrix_tuning_b200.optim import SMTAdam
    from sparse_matrix_tuning_b200.smt import smt as M, smt_helper as H
    w = torch.nn.Parameter(torch.zeros(256, 256))
    with pytest.raises(SMTLibraryError):
        M.LinearLayer_MatrixSparsity(w, index_list=[(0, 0)])
    with pytest.raises(SMTLibraryError):
        H.select_submatrix_based_on_grads({("q_proj", 0): torch.zeros(256, 256)}, {"q_proj": [256, 256]}, 1)
    with pytest.raises(SMTLibraryError):
        ops.score_accumulate(torch.zeros(8), torch.zeros(8))
    with pytest.raises(SMTLibraryError):
        SMTAdam([w])
    with pytest.raises((UnboundLocalError, ValueError)):
        H.select_submatrix_based_on_grads({}, {}, 1, calculate_strategy="bogus")


def test_index_table_cache_follows_the_list_by_value():
    """ops.index_table: one cache of index-list snapshots and the device tables derived from them, keyed on the list
    object and checked by value on every call."""
    from sparse_matrix_tuning_b200 import ops
    idx = [(0, 1), (2, 3)]
    snap, rc = ops.index_table(idx, ops.make_block_rc, "cpu")
    assert snap == ((0, 1), (2, 3)) and rc.tolist() == [[0, 1], [2, 3]]
    assert ops.index_table(idx, ops.make_block_rc, "cpu")[1] is rc               # same list, same contents
    assert ops.index_table(idx)[0] is snap
    idx[1] = (4, 5)                                                             # edited in place
    snap2, rc2 = ops.index_table(idx, ops.make_block_rc, "cpu")
    assert snap2 == ((0, 1), (4, 5)) and rc2 is not rc and rc2.tolist() == [[0, 1], [4, 5]]
    idx.append((6, 7))
    assert ops.index_table(idx, ops.make_block_rc, "cpu")[1].tolist() == [[0, 1], [4, 5], [6, 7]]
    twin = [list(e) for e in idx]                                               # equal, distinct, lists not tuples
    snap3, rc3 = ops.index_table(twin, ops.make_block_rc, "cpu")
    assert snap3 == ((0, 1), (4, 5), (6, 7)) and rc3.tolist() == [[0, 1], [4, 5], [6, 7]]
    assert ops.index_table(twin, ops.make_block_rc, "cpu")[1] is rc3
    # a different kind (builder or its arguments) or device is a separate entry of the same list
    ch = [5, 3, 9]
    plain = ops.index_table(ch, ops.make_channel_idx, "cpu", 1)[1]
    padded = ops.index_table(ch, ops.make_channel_idx, "cpu", 8)[1]
    meta = ops.index_table(ch, ops.make_channel_idx, "meta", 8)[1]
    assert plain.tolist() == [5, 3, 9] and padded.tolist() == [5, 3, 9] + [-1] * 5
    assert meta.device.type == "meta" and meta.shape == (8,)
    assert ops.index_table(ch, ops.make_channel_idx, "cpu", 1)[1] is plain
    assert ops.index_table(ch, ops.make_channel_idx, "cpu", 8)[1] is padded
    assert ops.index_table(ch, ops.make_channel_idx, "meta", 8)[1] is meta
    # bounded
    lists = [[i] for i in range(ops._INDEX_CACHE_MAX + 10)]
    for i, lst in enumerate(lists):
        assert ops.index_table(lst, ops.make_channel_idx, "cpu", 1)[1].tolist() == [i]
    assert len(ops._index_cache) <= ops._INDEX_CACHE_MAX


def test_no_oracle_import_in_product_package():
    pkg = os.path.join(ROOT, "sparse_matrix_tuning_b200")
    for dirpath, _d, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "/root/reference" not in src, f


def test_reference_driver_import_lines_resolve_to_this_package():
    """INTEGRATION.md §1: with <repo> and <repo>/sparse_matrix_tuning_b200 on PYTHONPATH, the exact import lines of the
    reference driver (fine_tune.py:39-40) pick up the mirror package."""
    import subprocess
    import sys
    code = (
        "from smt.smt import convert_linear_layer_to_matrix_sparsity, get_optimizer_sparse_grouped_parameters, "
        "get_optimizer_qk_augment_grouped_parameters, freeze_unselected_matrix_layer, freeze_unselected_channel_layer, "
        "convert_linear_layer_to_channel_sparsity\n"
        "from smt.smt_helper import select_submatrix_based_on_grads, get_blocks, get_named_linears, "
        "select_channel_based_on_activation\n"
        "import smt.smt as S\n"
        "import sparse_matrix_tuning_b200.smt.smt as C, sparse_matrix_tuning_b200.optim\n"
        "assert S is C and convert_linear_layer_to_matrix_sparsity is C.convert_linear_layer_to_matrix_sparsity\n"
        "print(S.__file__)\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "sparse_matrix_tuning_b200")]))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd="/tmp", timeout=300)
    assert out.returncode == 0, out.stderr
    assert os.path.join("sparse_matrix_tuning_b200", "smt", "smt.py") in out.stdout


def test_block_budget_helpers_match_the_reference_golden():
    """a-3: the PRODUCT helpers `smt_helper.targeted_module_dims / num_total_blocks / block_budget` restate the driver's
    inline arithmetic (fine_tune.py:217-241) and must reproduce the numbers the reference-generated config-1 golden
    holds: 596 blocks in total (embeddings and lm_head included), int(0.01 * 596) = 5, and the dims dict."""
    from conftest import load_golden
    from oracle import golden_inputs as GI
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    gold = load_golden("config1_e2e.pt")
    model, _batches = GI.make_config1()
    assert H.num_total_blocks(model) == gold["total_blocks"] == 596
    assert H.block_budget(model, GI.CONFIG1["attn_ratio"]) == gold["n_attn"] == 5
    assert H.targeted_module_dims(model) == gold["dims"]
    assert H.block_budget(model, 0.0084) == int(0.0084 * 596)            # truncation, not rounding (fine_tune.py:236)
    assert H.block_budget(model, 0.01, block=128) == int(0.01 * 596 * 4)
    # LLaMA-3-8B: the figures BASELINE.md quotes, from shapes alone (meta tensors, nothing allocated)
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=128256, hidden_size=4096, intermediate_size=14336, num_hidden_layers=32,
                      num_attention_heads=32, num_key_value_heads=8, tie_word_embeddings=False)
    with torch.device("meta"):
        big = LlamaForCausalLM(cfg)
    assert H.num_total_blocks(big) == 122528 and H.block_budget(big, 0.0071) == 869 and H.block_budget(big, 0.0086) == 1053
    assert H.targeted_module_dims(big)["k_proj"] == [1024, 4096]

