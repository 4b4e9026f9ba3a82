"""CPU tests of the Mistral / Qwen3 support of the fused decoder path: argument validation of `smt_qk_norm_rope_*`
without a device, and which transformers classes `layer_supported` / `install_causal_lm` accept."""
import ctypes

import pytest
import torch


def _p(buf):
    return ctypes.cast(buf, ctypes.c_void_p).value


def _fwd(lib, q, k, wq, wk, cs, B, S, Hq, Hk, bstride, qo, ko, rq, rk):
    return lib.smt_qk_norm_rope_forward(q, k, wq, wk, 1e-6, 1e-6, cs, cs, B, S, Hq, Hk, bstride, qo, ko, rq, rk, None)


def _bwd(lib, q, k, wq, wk, rq, rk, cs, dqo, dko, B, S, Hq, Hk, bstride, dq, dk):
    return lib.smt_qk_norm_rope_backward(q, k, wq, wk, rq, rk, cs, cs, dqo, dko, B, S, Hq, Hk, bstride, dq, dk, None)


def test_qk_norm_rope_rejects_bad_arguments_without_a_device(built_library):
    lib = built_library
    buf = ctypes.create_string_buffer(8192 + 16)
    b = (_p(buf) + 15) & ~15
    # negative shapes and a cos/sin batch stride that is not a multiple of 8
    for shape in ((-1, 1, 1, 1, 0), (1, -1, 1, 1, 0), (1, 1, -1, 1, 0), (1, 1, 1, -1, 0), (1, 1, 1, 1, -8),
                  (2, 1, 1, 1, 12)):
        assert _fwd(lib, b, b, b, b, b, *shape, b, b, b, b) == -1
        assert b"bad shape" in lib.smt_last_error()
        assert _bwd(lib, b, b, b, b, b, b, b, b, b, *shape, b, b) == -1
        assert b"bad shape" in lib.smt_last_error()
    # every pointer of the forward, then of the backward, null in turn
    for i in range(9):
        args = [b] * 9
        args[i] = None
        q, k, wq, wk, cs, qo, ko, rq, rk = args
        assert _fwd(lib, q, k, wq, wk, cs, 1, 1, 1, 1, 0, qo, ko, rq, rk) == -1
        assert b"null pointer" in lib.smt_last_error()
    for i in range(11):
        args = [b] * 11
        args[i] = None
        q, k, wq, wk, rq, rk, cs, dqo, dko, dq, dk = args
        assert _bwd(lib, q, k, wq, wk, rq, rk, cs, dqo, dko, 1, 1, 1, 1, 0, dq, dk) == -1
        assert b"null pointer" in lib.smt_last_error()
    # a tensor off the 16-byte grid (rstd off the 4-byte grid)
    for i in range(7):
        args = [b] * 7
        args[i] = b + 2
        q, k, wq, wk, cs, qo, ko = args
        assert _fwd(lib, q, k, wq, wk, cs, 1, 1, 1, 1, 0, qo, ko, b, b) == -1
        assert b"aligned" in lib.smt_last_error()
    assert _fwd(lib, b, b, b, b, b, 1, 1, 1, 1, 0, b, b, b + 2, b) == -1
    assert b"aligned" in lib.smt_last_error()
    assert _bwd(lib, b + 8, b, b, b, b, b, b, b, b, 1, 1, 1, 1, 0, b, b) == -1
    assert b"aligned" in lib.smt_last_error()
    # no rows is a no-op, even with null pointers; a side without rows needs no pointers
    assert _fwd(lib, None, None, None, None, None, 0, 4, 2, 1, 0, None, None, None, None) == 0
    assert _fwd(lib, None, None, None, None, None, 2, 4, 0, 0, 0, None, None, None, None) == 0
    assert _bwd(lib, None, None, None, None, None, None, None, None, None, 1, 0, 2, 1, 0, None, None) == 0


def test_qk_norm_rope_op_needs_cuda(built_library):
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    q = torch.zeros(1, 2, 2, 128, dtype=torch.bfloat16)
    k = torch.zeros(1, 2, 1, 128, dtype=torch.bfloat16)
    w = torch.ones(128, dtype=torch.bfloat16)
    cs = torch.zeros(1, 2, 128, dtype=torch.bfloat16)
    with pytest.raises(SMTLibraryError):
        ops.qk_norm_rope_forward(q, k, w, w, 1e-6, 1e-6, cs, cs)


# ---- which classes the overrides accept ----------------------------------------------------------------------------

_SMALL = dict(vocab_size=64, hidden_size=256, intermediate_size=512, num_hidden_layers=1, num_attention_heads=2,
              num_key_value_heads=1, head_dim=128, max_position_embeddings=64)


def _model(family, **kw):
    import transformers
    cfg = getattr(transformers, f"{family}Config")(**{**_SMALL, **kw})
    torch.manual_seed(0)
    return getattr(transformers, f"{family}ForCausalLM")(cfg)


@pytest.mark.parametrize("family", ["Llama", "Mistral", "Qwen3"])
def test_supported_families_are_accepted(built_library, family):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    model = _model(family)
    layer = model.model.layers[0]
    assert D.layer_supported(layer)
    assert D.install_layer(layer) and D.install_norm(model.model.norm)
    if family == "Qwen3":
        # the per-head norms run inside the attention override's kernel, never through the RMSNorm override
        assert "forward" not in layer.self_attn.q_norm.__dict__ and "forward" not in layer.self_attn.k_norm.__dict__
    assert D.remove_all(model) == 1
    assert D.install_causal_lm(model) and D.remove_causal_lm(model)


def test_unsupported_layers_and_models_are_rejected(built_library):
    import transformers
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.smt import smt as M
    # Qwen3 with head_dim 64 (q_norm / k_norm of width 64)
    narrow = _model("Qwen3", head_dim=64, num_attention_heads=4, num_key_value_heads=2)
    assert not D.layer_supported(narrow.model.layers[0])
    # a subclass of a supported class
    from transformers.models.qwen3.modeling_qwen3 import Qwen3DecoderLayer

    class MyLayer(Qwen3DecoderLayer):
        pass
    model = _model("Qwen3")
    assert not D.layer_supported(MyLayer(model.config, 0))
    # Qwen2 (q/k/v biases): a different family
    qwen2 = transformers.Qwen2ForCausalLM(transformers.Qwen2Config(**{k: v for k, v in _SMALL.items()
                                                                        if k != "head_dim"}))
    assert not D.layer_supported(qwen2.model.layers[0])
    assert not D.install_causal_lm(qwen2) and not M.fuse_causal_lm_loss(qwen2)
    # a Qwen3Model is not a causal LM
    assert not D.install_causal_lm(model.model) and "forward" not in model.model.__dict__
    assert M.fuse_causal_lm_loss(model) and M.unfuse_causal_lm_loss(model)


@pytest.mark.parametrize("family", ["Mistral", "Qwen3"])
def test_cpu_calls_of_a_fused_model_run_the_class_forward(built_library, family):
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.smt import smt as M
    model = _model(family)
    for p in model.parameters():
        p.requires_grad_(False)
    ids = torch.randint(0, 64, (2, 8), generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        ref = model(input_ids=ids, labels=ids, use_cache=False)
        assert M.fuse_causal_lm_loss(model)
        assert all(D.install_layer(l) for l in model.model.layers) and D.install_norm(model.model.norm)
        got = model(input_ids=ids, labels=ids, use_cache=False)
    assert torch.equal(got.loss, ref.loss) and torch.equal(got.logits, ref.logits)
