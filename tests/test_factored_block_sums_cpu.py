"""CPU tests of the factored warm-up block sums: argument validation of `smt_token_block_sums` and
`smt_block_outer_accumulate` without a device, the ops' refusal of CPU tensors, `FactoredBlockSumAccumulator`'s hooks on
a tiny LLaMA, and the world-2 `gloo` block-sum all-reduce with the new accumulator."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _p(buf):
    return ctypes.cast(buf, ctypes.c_void_p).value


def test_token_block_sums_rejects_bad_arguments_without_a_device(built_library):
    lib = built_library
    buf = ctypes.create_string_buffer(8192 + 16)
    base = (_p(buf) + 15) & ~15
    F32, BF16 = 0, 1
    # T = 0 (or F = 0) is a no-op, even with null pointers
    assert lib.smt_token_block_sums(None, BF16, 0, 256, 256, 256, None, None) == 0
    assert lib.smt_token_block_sums(None, BF16, 4, 0, 0, 64, None, None) == 0
    # negative sizes
    assert lib.smt_token_block_sums(base, BF16, -1, 256, 256, 256, base, None) == -1
    assert b"negative" in lib.smt_last_error()
    assert lib.smt_token_block_sums(base, BF16, 1, -256, 256, 256, base, None) == -1
    # bad dtype, bad block, F not a multiple of the block
    assert lib.smt_token_block_sums(base, 3, 1, 256, 256, 256, base, None) == -1
    assert b"dtype" in lib.smt_last_error()
    assert lib.smt_token_block_sums(base, BF16, 1, 256, 256, 32, base, None) == -1
    assert b"block" in lib.smt_last_error()
    assert lib.smt_token_block_sums(base, BF16, 1, 320, 320, 256, base, None) == -1
    assert b"multiple" in lib.smt_last_error()
    # null pointers
    assert lib.smt_token_block_sums(None, BF16, 1, 256, 256, 256, base, None) == -1
    assert b"null pointer" in lib.smt_last_error()
    assert lib.smt_token_block_sums(base, BF16, 1, 256, 256, 256, None, None) == -1
    # row pitch below F, or not a multiple of 16 bytes; misaligned bases
    assert lib.smt_token_block_sums(base, BF16, 2, 256, 128, 64, base, None) == -1
    assert lib.smt_token_block_sums(base, BF16, 2, 256, 260, 64, base, None) == -1
    assert lib.smt_token_block_sums(base, F32, 2, 256, 258, 64, base, None) == -1
    assert lib.smt_token_block_sums(base + 2, BF16, 2, 256, 256, 64, base, None) == -1
    assert b"aligned" in lib.smt_last_error()
    assert lib.smt_token_block_sums(base, BF16, 2, 256, 256, 64, base + 2, None) == -1
    assert b"aligned" in lib.smt_last_error()


def test_block_outer_accumulate_rejects_bad_arguments_without_a_device(built_library):
    lib = built_library
    buf = ctypes.create_string_buffer(8192 + 16)
    base = (_p(buf) + 15) & ~15
    assert lib.smt_block_outer_accumulate_workspace_bytes(0, 4, 4) == 0
    assert lib.smt_block_outer_accumulate_workspace_bytes(1, 4, 4) == 64
    assert lib.smt_block_outer_accumulate_workspace_bytes(128, 16, 56) == 16 * 56 * 4      # fixed 128-token chunks
    assert lib.smt_block_outer_accumulate_workspace_bytes(129, 16, 56) == 2 * 16 * 56 * 4
    ws = lib.smt_block_outer_accumulate_workspace_bytes(8, 2, 2)
    # T = 0 is a no-op, even with null pointers
    assert lib.smt_block_outer_accumulate(None, None, None, 0, 2, 2, None, 0, None) == 0
    # negative sizes
    for T, rb, cb in ((-1, 2, 2), (8, -2, 2), (8, 2, -2)):
        assert lib.smt_block_outer_accumulate(base, base, base, T, rb, cb, base, ws, None) == -1
        assert b"negative" in lib.smt_last_error()
    # null pointers
    for i in range(4):
        ptrs = [base] * 4
        ptrs[i] = None
        acc, dy, x, w = ptrs
        assert lib.smt_block_outer_accumulate(acc, dy, x, 8, 2, 2, w, ws, None) == -1
        assert b"null pointer" in lib.smt_last_error()
    # misaligned fp32 arrays
    for i in range(4):
        ptrs = [base] * 4
        ptrs[i] = base + 2
        acc, dy, x, w = ptrs
        assert lib.smt_block_outer_accumulate(acc, dy, x, 8, 2, 2, w, ws, None) == -1
        assert b"aligned" in lib.smt_last_error()
    # workspace too small
    assert lib.smt_block_outer_accumulate(base, base, base, 8, 2, 2, base, ws - 4, None) == -4


def test_ops_need_cuda(built_library):
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    with pytest.raises(SMTLibraryError):
        ops.token_block_sums(torch.zeros(4, 256, dtype=torch.bfloat16), 256)
    with pytest.raises(SMTLibraryError):
        ops.block_outer_accumulate(torch.zeros(2, 3), torch.zeros(4, 2), torch.zeros(4, 3))


def _tiny_llama(hidden=256, inter=512, vocab=64):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=vocab, hidden_size=hidden, intermediate_size=inter, num_hidden_layers=2,
                      num_attention_heads=2, num_key_value_heads=2, max_position_embeddings=32)
    torch.manual_seed(0)
    return LlamaForCausalLM(cfg)


def _hooked(model):
    return sorted(n for n, m in model.named_modules() if isinstance(m, torch.nn.Linear) and m._forward_hooks)


def test_attach_hooks_exactly_the_targeted_modules_and_detach_removes_them(built_library):
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    model = _tiny_llama()
    before = {n: dict(m._forward_hooks) for n, m in model.named_modules()}
    acc = FactoredBlockSumAccumulator(block=256)
    assert acc.attach(model) is acc
    assert _hooked(model) == sorted(f"model.layers.{l}.self_attn.{k}" for l in range(2)
                                    for k in ("q_proj", "k_proj", "v_proj"))
    assert list(acc.acc) == [(k, l) for l in range(2) for k in ("q_proj", "k_proj", "v_proj")]   # module order
    assert acc.shapes[("q_proj", 0)] == (256, 256) and acc.acc[("k_proj", 1)].shape == (1, 1)
    acc.detach()
    assert {n: dict(m._forward_hooks) for n, m in model.named_modules()} == before
    mlp = FactoredBlockSumAccumulator(block=256, mlp=True).attach(model)
    hooked = _hooked(model)
    assert not any("o_proj" in n for n in hooked) and len(hooked) == 12
    assert {k for k, _l in mlp.acc} == {"q_proj", "k_proj", "v_proj", "gate_proj", "up_proj", "down_proj"}
    assert mlp.acc[("down_proj", 0)].shape == (1, 2)
    mlp.detach()
    only_mlp = FactoredBlockSumAccumulator(block=256, mlp=True, attention=False).attach(model)
    assert {k for k, _l in only_mlp.acc} == {"gate_proj", "up_proj", "down_proj"}
    only_mlp.detach()
    assert {n: dict(m._forward_hooks) for n, m in model.named_modules()} == before


def test_attach_rejects_features_that_are_not_multiples_of_the_block(built_library):
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    model = _tiny_llama(hidden=256, inter=320)
    FactoredBlockSumAccumulator(block=64, mlp=True).attach(model).detach()
    acc = FactoredBlockSumAccumulator(block=256, mlp=True)
    with pytest.raises(SMTLibraryError, match="mlp"):
        acc.attach(model)
    assert _hooked(model) == []


def test_cpu_forward_raises_and_no_grad_forward_does_nothing(built_library):
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    model = _tiny_llama()
    for p in model.parameters():
        p.requires_grad_(False)
    model.enable_input_require_grads()
    acc = FactoredBlockSumAccumulator(block=256).attach(model)
    ids = torch.randint(0, 64, (1, 8))
    with torch.no_grad():
        model(input_ids=ids, use_cache=False)
    assert all(not t.any() for t in acc.acc.values()) and acc._x_cache is None
    with pytest.raises(SMTLibraryError):
        model(input_ids=ids, use_cache=False)
    acc.detach()


def test_scores_accept_mean_abs_only(built_library):
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    acc = FactoredBlockSumAccumulator()
    for strategy in ("abs_mean", "L1", "L2"):
        with pytest.raises(SMTLibraryError):
            acc.scores(strategy)


def test_flat_state_round_trip():
    from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
    acc = FactoredBlockSumAccumulator()
    acc.acc = {("q_proj", 0): torch.arange(4.0).view(2, 2), ("k_proj", 0): torch.arange(2.0).view(1, 2)}
    flat = acc.flat_state()
    assert torch.equal(flat, torch.tensor([0.0, 1.0, 2.0, 3.0, 0.0, 1.0]))
    acc.load_flat_state(flat * 2)
    assert torch.equal(acc.acc[("q_proj", 0)], torch.arange(4.0).view(2, 2) * 2)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, results):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from sparse_matrix_tuning_b200 import dp
        from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator
        acc = FactoredBlockSumAccumulator(block=256)
        acc.acc = {("q_proj", 0): torch.full((2, 2), float(rank + 1)),
                   ("k_proj", 0): torch.full((1, 2), 10.0 * (rank + 1))}
        dp.allreduce_block_sums(acc)                        # block sums of the data-parallel MEAN gradient
        assert torch.equal(acc.acc[("q_proj", 0)], torch.full((2, 2), 1.5))
        assert torch.equal(acc.acc[("k_proj", 0)], torch.full((1, 2), 15.0))
        results[rank] = "ok"
    except Exception as e:  # pragma: no cover
        results[rank] = f"{type(e).__name__}: {e}"
    finally:
        dist.destroy_process_group()


def test_allreduce_block_sums_takes_the_factored_accumulator():
    world = 2
    port = _free_port()
    with mp.Manager() as mgr:
        results = mgr.dict()
        mp.spawn(_worker, args=(world, port, results), nprocs=world, join=True)
        assert dict(results) == {0: "ok", 1: "ok"}
