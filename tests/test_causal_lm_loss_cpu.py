"""CPU tests of the fused lm_head + causal-LM loss: argument validation of `smt_cross_entropy_rows` without a device,
and installation of the `LlamaForCausalLM` override (class and signature guard, removal, CPU calls run the class's own
forward)."""
import copy
import ctypes

import pytest
import torch


def _p(buf):
    return ctypes.cast(buf, ctypes.c_void_p).value


def test_cross_entropy_rows_rejects_bad_arguments_without_a_device(built_library):
    lib = built_library
    buf = ctypes.create_string_buffer(4096 + 16)
    base = (_p(buf) + 15) & ~15
    # V % 8 != 0
    assert lib.smt_cross_entropy_rows(base, 8, 1, 12, base, -100, base, base, None) == -1
    assert b"V = 12" in lib.smt_last_error()
    # row pitch below V, or not a multiple of 8
    assert lib.smt_cross_entropy_rows(base, 8, 1, 16, base, -100, base, base, None) == -1
    assert lib.smt_cross_entropy_rows(base, 20, 1, 16, base, -100, base, base, None) == -1
    # null pointers
    for i in range(4):
        ptrs = [base] * 4
        ptrs[i] = None
        logits, labels, scale, loss = ptrs
        assert lib.smt_cross_entropy_rows(logits, 16, 2, 16, labels, -100, scale, loss, None) == -1
        assert b"null pointer" in lib.smt_last_error()
    # misaligned logits
    assert lib.smt_cross_entropy_rows(base + 2, 16, 2, 16, base, -100, base, base, None) == -1
    # negative row count
    assert lib.smt_cross_entropy_rows(base, 16, -1, 16, base, -100, base, base, None) == -1
    # T = 0 is a no-op, even with null pointers
    assert lib.smt_cross_entropy_rows(None, 16, 0, 16, None, -100, None, None, None) == 0


def test_cross_entropy_rows_op_needs_cuda(built_library):
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    with pytest.raises(SMTLibraryError):
        ops.cross_entropy_rows(torch.zeros(2, 16, dtype=torch.bfloat16), torch.zeros(2, dtype=torch.int64),
                               torch.ones(1))


def _tiny_llama():
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=64, hidden_size=32, intermediate_size=64, num_hidden_layers=1, num_attention_heads=2,
                      num_key_value_heads=1, max_position_embeddings=32)
    torch.manual_seed(0)
    return LlamaForCausalLM(cfg)


def test_fuse_causal_lm_loss_installs_on_llama_only(built_library):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.smt import smt as M
    model = _tiny_llama()
    assert not M.unfuse_causal_lm_loss(model)
    assert not M.fuse_causal_lm_loss(model.model)               # a LlamaModel is not a LlamaForCausalLM
    assert M.fuse_causal_lm_loss(model)
    assert model.__dict__["forward"].__func__ is D._causal_lm_forward
    twin = copy.deepcopy(model)
    assert twin.__dict__["forward"].__self__ is twin
    assert M.unfuse_causal_lm_loss(model) and "forward" not in model.__dict__
    assert not M.unfuse_causal_lm_loss(model)
    # unfusing the decoder layers leaves the loss override alone
    M.unfuse_qkv_projections(twin)
    assert twin.__dict__["forward"].__func__ is D._causal_lm_forward


def test_cpu_calls_run_the_class_forward(built_library):
    from sparse_matrix_tuning_b200.smt import smt as M
    model = _tiny_llama()
    for p in model.lm_head.parameters():
        p.requires_grad_(False)
    ids = torch.randint(0, 64, (2, 8))
    ref = model(input_ids=ids, labels=ids, use_cache=False)
    M.fuse_causal_lm_loss(model)
    got = model(input_ids=ids, labels=ids, use_cache=False)
    assert torch.equal(got.loss, ref.loss) and torch.equal(got.logits, ref.logits)
    tup = model(input_ids=ids, labels=ids, use_cache=False, return_dict=False)
    assert isinstance(tup, tuple) and torch.equal(tup[0], ref.loss)
