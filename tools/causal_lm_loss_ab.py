"""A/B of the fused lm_head + causal-LM loss (csrc/loss_kernels.cu, decoder_fusion.LinearCrossEntropyFn) against
transformers' `lm_head` + `ForCausalLMLoss`, on one GPU, in one process; prints one JSON object (and writes it to --out).

  1. the row kernel at T tokens, V = 128 256: CUDA events around each launch (median of --iters), fresh logits copied
     in and a 256 MB memset before each launch so that the 2.1 GB of logits come from HBM and not from the 126 MB L2;
     GB/s counting 4 bytes per logit (one bf16 read, one bf16 write) and the fraction of --hbm-gbs;
  2. lm_head + loss, forward + backward, at LLaMA-3-8B widths and T tokens: fused (chunk of {1024, 2048, 4096, 8192}
     rows) against HF, alternated, with peak memory above the inputs;
  3. the whole SMT step of bench.py's shape (tools/decoder_fusion_ab.py `whole_step`, q/k/v and decoder fusion on in
     both arms): fused loss on against off, alternating, with ms/step and max_memory_allocated per arm.

    python tools/causal_lm_loss_ab.py --out /tmp/r04_causal_lm_loss_raw.json
    python tools/causal_lm_loss_ab.py --dry-run          # shapes and byte counts only, no GPU
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from decoder_fusion_ab import HID, LLAMA3_8B, NKV, HD, gpu_info  # noqa: E402

VOCAB = LLAMA3_8B["vocab_size"]
CHUNKS = (1024, 2048, 4096, 8192)


def kernel_bytes(T: int) -> int:
    return 4 * T * VOCAB


def per_kernel(T, iters, hbm_gbs):
    import torch
    from sparse_matrix_tuning_b200 import ops
    torch.manual_seed(0)
    src = (torch.randn(T, VOCAB, device="cuda") * 3).bfloat16()
    logits = torch.empty_like(src)
    y = torch.randint(0, VOCAB, (T,), device="cuda")
    scale = torch.full((1,), 1.0 / T, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ts = []
    for i in range(iters + 3):
        logits.copy_(src)
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.cross_entropy_rows(logits, y, scale, -100)
        b.record()
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(a.elapsed_time(b))
    ms = statistics.median(ts)
    gbs = kernel_bytes(T) / (ms * 1e-3) / 1e9
    return {"us": ms * 1e3, "us_min": min(ts) * 1e3, "bytes": kernel_bytes(T), "gb_per_s": gbs,
            "fraction_of_hbm_peak": gbs / hbm_gbs}


def lm_head_loss(T, iters):
    """Forward + backward of lm_head + loss from the final-norm output h [T, 4096], frozen W [128256, 4096]."""
    import torch
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    torch.manual_seed(0)
    h = torch.randn(T, HID, device="cuda").bfloat16()
    w = (torch.randn(VOCAB, HID, device="cuda") * 0.02).bfloat16()
    labels = torch.randint(0, VOCAB, (1, T), device="cuda")

    def fused():
        hg = h.clone().requires_grad_(True)
        D.causal_lm_loss(hg, w, labels).backward()

    def hf():
        hg = h.clone().requires_grad_(True)
        ForCausalLMLoss(torch.nn.functional.linear(hg, w)[None], labels, VOCAB).backward()

    def measure(fn):
        fn()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        ts = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts), peak

    default = D._CE_CHUNK_ROWS
    res = {"hf": {"ms": [], "peak_bytes_above_inputs": 0}}
    try:
        for _rep in range(2):
            for c in CHUNKS:
                D._CE_CHUNK_ROWS = c
                ms, peak = measure(fused)
                r = res.setdefault(f"fused_chunk{c}", {"ms": [], "peak_bytes_above_inputs": 0})
                r["ms"].append(ms)
                r["peak_bytes_above_inputs"] = max(r["peak_bytes_above_inputs"], peak)
                ms, peak = measure(hf)
                res["hf"]["ms"].append(ms)
                res["hf"]["peak_bytes_above_inputs"] = max(res["hf"]["peak_bytes_above_inputs"], peak)
    finally:
        D._CE_CHUNK_ROWS = default
    for r in res.values():
        r["ms_min"] = min(r["ms"])
        r["ms_median"] = statistics.median(r["ms"])
    return {"tokens": T, "arms": res, "default_chunk_rows": default}


def whole_step(steps, reps, batch, seq):
    """bench.py's SMT step at its default shape, q/k/v and decoder fusion on in both arms: fused loss on / off."""
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.optim import SMTAdam
    from sparse_matrix_tuning_b200.smt import smt as M
    cfg = LlamaConfig(**LLAMA3_8B)
    torch.manual_seed(1234)
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device("cuda"):
            model = LlamaForCausalLM(cfg)
    finally:
        torch.set_default_dtype(torch.float32)
    model.config.use_cache = False
    rng = random.Random(0)
    sel = {}
    shapes = {"q_proj": (HID // 256, HID // 256), "k_proj": (NKV * HD // 256, HID // 256),
              "v_proj": (NKV * HD // 256, HID // 256)}
    cand = [(kind, l, r, c) for l in range(32) for kind, (R, C) in shapes.items() for r in range(R) for c in range(C)]
    for kind, l, r, c in sorted(rng.sample(cand, 869)):
        sel.setdefault((kind, l), []).append((r, c))
    M.freeze_unselected_matrix_layer(model, {}, sel)
    M.convert_linear_layer_to_matrix_sparsity(model, {}, sel)
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    model.train()
    opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-4), lr=1e-4, betas=(0.9, 0.95),
                  max_grad_norm=1.0)
    M.set_grouped_backward(True)
    M.fuse_qkv_projections(model)
    gen = torch.Generator().manual_seed(0)
    ids = [torch.randint(0, cfg.vocab_size, (batch, seq), generator=gen).cuda() for _ in range(steps)]

    def step(t):
        loss = model(input_ids=t, labels=t, use_cache=False).loss
        loss.backward()
        opt.step()
        opt.zero_grad()
        return loss

    res = {"fused_loss": [], "hf_loss": []}
    per_step = {"fused_loss": [], "hf_loss": []}
    peak = {"fused_loss": 0, "hf_loss": 0}
    for _ in range(reps):
        for arm in ("fused_loss", "hf_loss"):
            if arm == "fused_loss":
                assert M.fuse_causal_lm_loss(model)
            # each arm starts from an empty allocator cache, not from the blocks the other arm's tensors left behind
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            for i in range(2):
                step(ids[i])
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            ev[0].record()
            for t, e in zip(ids, ev[1:]):
                step(t)
                e.record()
            torch.cuda.synchronize()
            peak[arm] = max(peak[arm], torch.cuda.max_memory_allocated())
            res[arm].append(ev[0].elapsed_time(ev[-1]) / steps)
            per_step[arm].append([a.elapsed_time(b) for a, b in zip(ev[:-1], ev[1:])])
            M.unfuse_causal_lm_loss(model)
    M.unfuse_qkv_projections(model)
    M.set_grouped_backward(False)
    return {"ms_per_step": res, "ms_each_step": per_step, "max_memory_allocated_bytes": peak,
            "steps_per_rep": steps, "reps": reps,
            "tokens_per_step": batch * seq,
            "speedup_min_over_pairs": min(u / f for u, f in zip(res["hf_loss"], res["fused_loss"])),
            "speedup_max_over_pairs": max(u / f for u, f in zip(res["hf_loss"], res["fused_loss"])),
            "ms_min_per_arm": {k: min(v) for k, v in res.items()},
            "peak_saving_bytes": peak["hf_loss"] - peak["fused_loss"], "chunk_rows": D._CE_CHUNK_ROWS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--op-iters", type=int, default=5)
    ap.add_argument("--steps", type=int, default=8, help="timed steps per arm and repetition of the whole step")
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--hbm-gbs", type=float, default=6545.6, help="HBM bandwidth the fractions refer to")
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--out", default="")
    ap.add_argument("--dry-run", action="store_true", help="print the shapes and byte counts, touch no GPU")
    args = ap.parse_args()
    if args.tokens % 512:
        raise SystemExit("--tokens must be a multiple of 512 (sequences of 512)")
    if args.dry_run:
        print(json.dumps({"tokens": args.tokens, "vocab": VOCAB, "kernel_bytes": kernel_bytes(args.tokens),
                          "chunks": CHUNKS}))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    t0 = time.time()
    result = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "tokens": args.tokens, "vocab": VOCAB,
              "hbm_gbs_reference": args.hbm_gbs, "l2_flush_bytes_between_launches": 256 << 20}
    result["kernel"] = per_kernel(args.tokens, args.iters, args.hbm_gbs)
    torch.cuda.empty_cache()
    result["lm_head_loss_fwd_bwd"] = lm_head_loss(args.tokens, args.op_iters)
    torch.cuda.empty_cache()
    if not args.skip_step:
        result["whole_step"] = whole_step(args.steps, args.reps, 16, 512)
    result["wall_s"] = time.time() - t0
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
