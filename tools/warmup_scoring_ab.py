"""A/B of the warm-up scoring pass: factored block sums on a frozen, fused model against the weight-gradient capture
`bench.py` runs, on one GPU, in one process; prints one JSON object (and writes it to --out).

  1. `token_block_sums` at T tokens, F in {1024, 4096, 14336}, bf16, b = 256: median of --iters CUDA-event timings,
     a 256 MB memset before each launch so the input comes from HBM and not from the 126 MB L2; GB/s counting one
     read of the input and one write of the fp32 sums, and the fraction of --hbm-gbs.  `block_outer_accumulate` at the
     q/k/v and MLP shapes is timed the same way (reported only).
  2. one warm-up pass (forward + backward) of LLaMA-3-8B, 32 layers, bf16, B 16 x S 512, non-reentrant recomputation,
     seeded random init, three arms alternated over --reps repetitions (--passes timed steady-state passes each):
       A  bench.py's pass: trainable q/k/v, WarmupGradAccumulator(block_sum).attach(free_grads=True), no fusion;
       B  frozen model, fuse_qkv_projections + fuse_causal_lm_loss, FactoredBlockSumAccumulator;
       C  B without hooks.
     Then the same three arms with MLP scoring (gate/up/down as well, the config-5 shape).  max_memory_allocated per arm.
  3. agreement: Jaccard overlap of the top-869 q/k/v selection of A and B after two passes on the same batches, SDPA
     on the math backend (random-init scores are near-ties: reported, no bar).

    python tools/warmup_scoring_ab.py --out /tmp/r05_factored_block_sums_raw.json
    python tools/warmup_scoring_ab.py --dry-run          # shapes and byte counts only, no GPU
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from decoder_fusion_ab import LLAMA3_8B, gpu_info  # noqa: E402

BLOCK = 256
KERNEL_F = (1024, 4096, 14336)
N_ATTN = 869                      # int(0.0071 * 122 528), bench.py's q/k/v budget
KINDS_ATTN = ("q_proj", "k_proj", "v_proj")


def kernel_bytes(T: int, F: int) -> int:
    return 2 * T * F + 4 * T * (F // BLOCK)


def per_kernel(T, iters, hbm_gbs):
    import torch
    from sparse_matrix_tuning_b200 import ops
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts), min(ts)

    res = {}
    g = torch.Generator(device="cuda").manual_seed(0)
    for F in KERNEL_F:
        x = torch.randn(T, F, device="cuda", generator=g).bfloat16()
        ms, ms_min = timed(lambda: ops.token_block_sums(x, BLOCK))
        gbs = kernel_bytes(T, F) / (ms * 1e-3) / 1e9
        res[f"token_block_sums_F{F}"] = {"us": ms * 1e3, "us_min": ms_min * 1e3, "bytes": kernel_bytes(T, F),
                                         "gb_per_s": gbs, "fraction_of_hbm_peak": gbs / hbm_gbs}
        del x
    for rb, cb in ((16, 16), (4, 16), (56, 16), (16, 56)):
        d = torch.randn(T, rb, device="cuda", generator=g)
        x = torch.randn(T, cb, device="cuda", generator=g)
        acc = torch.zeros(rb, cb, device="cuda")
        ms, ms_min = timed(lambda: ops.block_outer_accumulate(acc, d, x))
        res[f"block_outer_accumulate_{rb}x{cb}"] = {"us": ms * 1e3, "us_min": ms_min * 1e3}
    return res


def build_model():
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(1234)
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device("cuda"):
            model = LlamaForCausalLM(LlamaConfig(**LLAMA3_8B))
    finally:
        torch.set_default_dtype(torch.float32)
    model.config.use_cache = False
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    model.train()
    return model


class Arms:
    """Switches one model between the three warm-up arms."""

    def __init__(self, model):
        self.model = model

    def setup(self, arm, mlp):
        """Returns the accumulators of the arm (attention, mlp or None), hooks attached."""
        from sparse_matrix_tuning_b200.smt import smt as M
        from sparse_matrix_tuning_b200.warmup import FactoredBlockSumAccumulator, WarmupGradAccumulator
        model = self.model
        M.unfuse_qkv_projections(model)
        M.unfuse_causal_lm_loss(model)
        if arm == "A":
            for name, p in model.named_parameters():
                p.requires_grad = (("self_attn" in name) and any(k in name for k in KINDS_ATTN)) or (mlp and "mlp" in name)
            acc_a = WarmupGradAccumulator(block=BLOCK, mode="block_sum", mlp=False, attention=True)
            acc_m = WarmupGradAccumulator(block=BLOCK, mode="block_sum", mlp=True, attention=False) if mlp else None
            for acc in (acc_a, acc_m):
                if acc is not None:
                    acc.attach(model, free_grads=True)
            return acc_a, acc_m
        for p in model.parameters():
            p.requires_grad = False
        assert M.fuse_qkv_projections(model) == LLAMA3_8B["num_hidden_layers"]
        assert M.fuse_causal_lm_loss(model)
        if arm == "C":
            return None, None
        acc_a = FactoredBlockSumAccumulator(block=BLOCK, mlp=False, attention=True).attach(model)
        acc_m = FactoredBlockSumAccumulator(block=BLOCK, mlp=True, attention=False).attach(model) if mlp else None
        return acc_a, acc_m

    @staticmethod
    def teardown(accs):
        for acc in accs:
            if acc is not None:
                acc.detach()


def one_pass(model, ids):
    model(input_ids=ids, labels=ids, use_cache=False).loss.backward()


def warmup_pass(model, ids, reps, passes):
    import torch
    arms = Arms(model)
    out = {}
    for mlp in (False, True):
        res = {a: [] for a in "ABC"}
        peak = {a: 0 for a in "ABC"}
        for _rep in range(reps):
            for arm in "ABC":
                accs = arms.setup(arm, mlp)
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
                one_pass(model, ids[0])                           # steady state: allocator and kernels warm
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                for i in range(passes):
                    t0 = time.perf_counter()
                    one_pass(model, ids[1 + i % 2])
                    torch.cuda.synchronize()
                    res[arm].append((time.perf_counter() - t0) * 1e3)
                peak[arm] = max(peak[arm], torch.cuda.max_memory_allocated())
                arms.teardown(accs)
                model.zero_grad(set_to_none=True)
        med = {a: statistics.median(v) for a, v in res.items()}
        out["mlp" if mlp else "qkv"] = {
            "ms_per_pass": res, "ms_median": med, "ms_min": {a: min(v) for a, v in res.items()},
            "max_memory_allocated_bytes": peak,
            "hook_cost_fraction_B_over_C": med["B"] / med["C"] - 1.0,
            "speedup_A_over_B": med["A"] / med["B"]}
    return out


def agreement(model, ids):
    import torch
    from torch.nn.attention import SDPBackend, sdpa_kernel
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    arms = Arms(model)
    sels = {}
    for arm in "AB":
        accs = arms.setup(arm, False)
        with sdpa_kernel(SDPBackend.MATH):
            for t in ids[:2]:
                one_pass(model, t)
        torch.cuda.synchronize()
        arms.teardown(accs)
        model.zero_grad(set_to_none=True)
        keys, scores = accs[0].scores("mean_abs")
        sel = H.select_submatrix_from_scores(keys, scores, N_ATTN, "no_restriction")
        sels[arm] = {(k, rc) for k, v in sel.items() for rc in v}
    a, b = sels["A"], sels["B"]
    return {"n_blocks": N_ATTN, "jaccard": len(a & b) / len(a | b), "common": len(a & b)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--passes", type=int, default=3, help="timed passes per arm and repetition")
    ap.add_argument("--hbm-gbs", type=float, default=6545.6, help="HBM bandwidth the fractions refer to")
    ap.add_argument("--skip-pass", action="store_true")
    ap.add_argument("--out", default="")
    ap.add_argument("--dry-run", action="store_true", help="print the shapes and byte counts, touch no GPU")
    args = ap.parse_args()
    if args.dry_run:
        print(json.dumps({"tokens": args.tokens, "kernel_bytes": {F: kernel_bytes(args.tokens, F) for F in KERNEL_F}}))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    t0 = time.time()
    result = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "tokens": args.tokens,
              "hbm_gbs_reference": args.hbm_gbs, "l2_flush_bytes_between_launches": 256 << 20}
    result["kernels"] = per_kernel(args.tokens, args.iters, args.hbm_gbs)
    torch.cuda.empty_cache()
    if not args.skip_pass:
        model = build_model()
        g = torch.Generator().manual_seed(1234)
        ids = [torch.randint(0, LLAMA3_8B["vocab_size"], (16, 512), generator=g).cuda() for _ in range(3)]
        result["warmup_pass"] = {"batch": 16, "seq": 512, "recompute": "non-reentrant", "passes": args.passes,
                                 "reps": args.reps, **warmup_pass(model, ids, args.reps, args.passes)}
        result["agreement_math_attention"] = agreement(model, ids)
    result["wall_s"] = time.time() - t0
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
