"""A/B of the decoder-layer elementwise kernels (csrc/decoder_kernels.cu) against the HF ops they replace, on one GPU,
in one process; prints one JSON object (and writes it to --out).

  1. per kernel, T tokens at LLaMA-3-8B widths: CUDA events around each launch (median of --iters), a 256 MB memset
     between launches so that the 64-235 MB operands come from HBM and not from the 126 MB L2; algorithmic bytes,
     GB/s and the fraction of --hbm-gbs;
  2. one LLaMA-3-8B decoder layer, forward + recompute + backward under non-reentrant checkpointing: elementwise
     fusion on vs off (q/k/v projections fused in both), with peak memory;
  3. the whole 32-layer SMT step (random block selection of bench.py's size, SMTAdam, grouped block gradients):
     elementwise fusion on vs off, q/k/v fused in both, alternating A B A B.

    python tools/decoder_fusion_ab.py --out /tmp/r03_decoder_fusion_raw.json
    python tools/decoder_fusion_ab.py --dry-run          # shapes and byte counts only, no GPU
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HID, INTER, NQ, NKV, HD = 4096, 14336, 32, 8, 128
LLAMA3_8B = dict(vocab_size=128256, hidden_size=HID, intermediate_size=INTER, num_hidden_layers=32,
                 num_attention_heads=NQ, num_key_value_heads=NKV, max_position_embeddings=8192, rms_norm_eps=1e-5,
                 rope_theta=500000.0, attn_implementation="sdpa")


def kernel_bytes(T: int) -> dict:
    """Bytes each kernel must move at least (bf16 tensors, fp32 rstd; weights and cos/sin tables are negligible)."""
    row, q_k = 2 * T * HID, 2 * T * (NQ + NKV) * HD
    mlp = 2 * T * INTER
    return {"rmsnorm_fwd": 2 * row + 4 * T,                      # x -> y, rstd
            "add_rmsnorm_fwd": 4 * row + 4 * T,                  # res, a -> h, y, rstd
            "rmsnorm_bwd_dres": 4 * row + 4 * T,                 # x, dy, dres, rstd -> dx
            "rope_fwd": 2 * q_k,                                 # q, k -> q, k
            "rope_bwd": 2 * q_k,
            "swiglu_fwd": 3 * mlp,                               # g, u -> h
            "swiglu_bwd": 5 * mlp}                               # g, u, dh -> dg, du


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [s.strip() for s in out[0].split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as e:  # reported, not fatal: the timings still carry the device name from torch
        return {"error": f"{type(e).__name__}: {e}"}


def time_ms(fn, iters, flush):
    """Median of CUDA-event times of `fn()`, the L2 overwritten by a memset before each timed launch."""
    import torch
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
    return statistics.median(ts)


def per_kernel(T, iters, hbm_gbs):
    import torch
    from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
    from sparse_matrix_tuning_b200 import ops
    dev, eps = "cuda", 1e-5
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.manual_seed(0)
    x = torch.randn(T, HID, device=dev).bfloat16()
    a = torch.randn(T, HID, device=dev).bfloat16()
    dy = torch.randn(T, HID, device=dev).bfloat16()
    w = (1 + 0.1 * torch.randn(HID, device=dev)).bfloat16()
    S = 512
    B = T // S
    q = torch.randn(B, S, NQ, HD, device=dev).bfloat16()
    k = torch.randn(B, S, NKV, HD, device=dev).bfloat16()
    pos = torch.arange(S, device=dev).float()[:, None] * (500000.0 ** (-torch.arange(0, HD, 2, device=dev) / HD))
    emb = torch.cat((pos, pos), -1)[None]
    cos, sin = emb.cos().bfloat16(), emb.sin().bfloat16()
    g = torch.randn(T, INTER, device=dev).bfloat16()
    u = torch.randn(T, INTER, device=dev).bfloat16()
    dh = torch.randn(T, INTER, device=dev).bfloat16()

    def hf_norm(t):
        tf = t.float()
        return w * (tf * torch.rsqrt(tf.pow(2).mean(-1, keepdim=True) + eps)).to(t.dtype)

    _y, rstd, _ = ops.rmsnorm_forward(x, w, eps)
    # HF backward graphs, built once (retain_graph) so that only the backward ops are timed
    xg = x.clone().requires_grad_(True)
    y_hf = hf_norm(xg)
    qg, kg = q.transpose(1, 2).requires_grad_(True), k.transpose(1, 2).requires_grad_(True)
    rq, rk = apply_rotary_pos_emb(qg, kg, cos, sin)
    gg, ug = g.clone().requires_grad_(True), u.clone().requires_grad_(True)
    h_hf = torch.nn.functional.silu(gg) * ug
    dq_o, dk_o = torch.randn_like(q), torch.randn_like(k)

    cases = {
        "rmsnorm_fwd": (lambda: ops.rmsnorm_forward(x, w, eps), lambda: hf_norm(x)),
        "add_rmsnorm_fwd": (lambda: ops.rmsnorm_forward(a, w, eps, res=x), lambda: hf_norm(x + a)),
        "rmsnorm_bwd_dres": (lambda: ops.rmsnorm_backward(x, w, rstd, dy, a),
                             lambda: torch.autograd.grad(y_hf, xg, dy, retain_graph=True)[0] + a),
        "rope_fwd": (lambda: ops.rope_forward(q, k, cos, sin),
                     lambda: apply_rotary_pos_emb(q.transpose(1, 2), k.transpose(1, 2), cos, sin)),
        "rope_bwd": (lambda: ops.rope_backward(dq_o, dk_o, cos, sin),
                     lambda: torch.autograd.grad((rq, rk), (qg, kg), (dq_o.transpose(1, 2), dk_o.transpose(1, 2)),
                                                 retain_graph=True)),
        "swiglu_fwd": (lambda: ops.swiglu_forward(g, u), lambda: torch.nn.functional.silu(g) * u),
        "swiglu_bwd": (lambda: ops.swiglu_backward(g, u, dh),
                       lambda: torch.autograd.grad(h_hf, (gg, ug), dh, retain_graph=True)),
    }
    nbytes = kernel_bytes(T)
    out = {}
    for name, (ours, hf) in cases.items():
        t_ours, t_hf = time_ms(ours, iters, flush), time_ms(hf, iters, flush)
        gbs = nbytes[name] / (t_ours * 1e-3) / 1e9
        out[name] = {"us": t_ours * 1e3, "hf_us": t_hf * 1e3, "speedup_vs_hf": t_hf / t_ours, "bytes": nbytes[name],
                     "gb_per_s": gbs, "fraction_of_hbm_peak": gbs / hbm_gbs}
    return out


def one_layer(T, iters):
    """One LLaMA-3-8B decoder layer, fwd + recompute + bwd (non-reentrant checkpoint), elementwise fusion on / off."""
    import torch
    from torch.utils.checkpoint import checkpoint
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer, LlamaRotaryEmbedding
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.smt import smt as M
    cfg = LlamaConfig(**{**LLAMA3_8B, "num_hidden_layers": 1})
    torch.manual_seed(0)
    torch.set_default_dtype(torch.bfloat16)
    try:
        layer = LlamaDecoderLayer(cfg, 0).cuda()
    finally:
        torch.set_default_dtype(torch.float32)
    for p in layer.parameters():
        p.requires_grad_(False)
    S = 512
    B = T // S
    x = torch.randn(B, S, HID, device="cuda").bfloat16().requires_grad_(True)
    dout = torch.randn(B, S, HID, device="cuda").bfloat16()
    pos = torch.arange(S, device="cuda")[None]
    pe = LlamaRotaryEmbedding(cfg).cuda()(x, pos)

    def step():
        out = checkpoint(lambda t: layer(t, position_embeddings=pe, position_ids=pos), x, use_reentrant=False)
        out.backward(dout)
        x.grad = None

    res = {}
    for arm in ("fused", "unfused", "fused", "unfused"):
        M.fuse_qkv_projections(layer)
        if arm == "unfused":
            D.remove_all(layer)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        step()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        ms = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        res.setdefault(arm, {"ms": [], "peak_bytes_above_inputs": peak})["ms"].append(statistics.median(ms))
        M.unfuse_qkv_projections(layer)
    for arm in res:
        res[arm]["ms_median_of_reps"] = statistics.median(res[arm]["ms"])
    res["speedup"] = res["unfused"]["ms_median_of_reps"] / res["fused"]["ms_median_of_reps"]
    return res


def whole_step(steps, reps, batch, seq):
    """The SMT step of bench.py at its default shape: fusion on / off alternating, q/k/v fused in both."""
    import random

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
    # ~869 q/k/v blocks, as bench.py's gradient-based selection picks at its default ratio
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
    gen = torch.Generator().manual_seed(0)
    ids = [torch.randint(0, cfg.vocab_size, (batch, seq), generator=gen).cuda() for _ in range(steps)]

    def step(t):
        loss = model(input_ids=t, labels=t, use_cache=False).loss
        loss.backward()
        opt.step()
        opt.zero_grad()
        return loss

    res = {"fused": [], "unfused": []}
    for _ in range(reps):
        for arm in ("fused", "unfused"):
            M.fuse_qkv_projections(model)
            if arm == "unfused":
                D.remove_all(model)
            for i in range(2):
                step(ids[i])
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for t in ids:
                step(t)
            b.record()
            torch.cuda.synchronize()
            res[arm].append(a.elapsed_time(b) / steps)
            M.unfuse_qkv_projections(model)
    M.set_grouped_backward(False)
    return {"ms_per_step": res, "steps_per_rep": steps, "reps": reps, "tokens_per_step": batch * seq,
            "speedup_min_over_pairs": min(u / f for u, f in zip(res["unfused"], res["fused"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--layer-iters", type=int, default=5)
    ap.add_argument("--steps", type=int, default=8, help="timed steps per arm and repetition of the whole step")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--hbm-gbs", type=float, default=6545.6, help="HBM bandwidth the fractions refer to")
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--out", default="")
    ap.add_argument("--dry-run", action="store_true", help="print the shapes and byte counts, touch no GPU")
    args = ap.parse_args()
    if args.tokens % 512:
        raise SystemExit("--tokens must be a multiple of 512 (sequences of 512)")
    if args.dry_run:
        print(json.dumps({"tokens": args.tokens, "bytes": kernel_bytes(args.tokens)}))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    t0 = time.time()
    result = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "tokens": args.tokens,
              "hbm_gbs_reference": args.hbm_gbs, "l2_flush_bytes_between_launches": 256 << 20}
    result["per_kernel"] = per_kernel(args.tokens, args.iters, args.hbm_gbs)
    torch.cuda.empty_cache()
    result["one_layer_fwd_recompute_bwd"] = one_layer(args.tokens, args.layer_iters)
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
