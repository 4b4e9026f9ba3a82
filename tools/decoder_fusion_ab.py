"""A/B of the decoder-layer elementwise kernels (csrc/decoder_kernels.cu) against the HF ops they replace, on one GPU,
in one process; prints one JSON object (and writes it to --out).

  1. per kernel, T tokens at LLaMA-3-8B widths: CUDA events around each launch (median of --iters), a 256 MB memset
     between launches so that the 64-235 MB operands come from HBM and not from the 126 MB L2; algorithmic bytes,
     GB/s and the fraction of --hbm-gbs;
  2. one LLaMA-3-8B decoder layer, forward + recompute + backward under non-reentrant checkpointing: elementwise
     fusion on vs off (q/k/v projections fused in both), with peak memory;
  3. the whole 32-layer SMT step (random block selection of bench.py's size, SMTAdam, grouped block gradients):
     elementwise fusion on vs off, q/k/v fused in both, alternating A B A B.

--family mistral / qwen3 runs the same at Mistral-7B-v0.3 / Qwen3-8B shapes.  For Qwen3 the per-kernel section adds the
per-head q/k RMSNorm + RoPE kernel against HF's q_norm + k_norm + apply_rotary_pos_emb and against the composition of
the existing kernels (smt_rmsnorm_* on [T*H, 128] rows, then smt_rope_*).  The whole step of these families selects
block_budget(model, 0.0071) q/k/v blocks and compares arm A (fuse_qkv_projections + fuse_causal_lm_loss) with arm B
(q/k/v GEMMs fused, elementwise ops and loss left to transformers), with max_memory_allocated per arm.

    python tools/decoder_fusion_ab.py --out /tmp/r03_decoder_fusion_raw.json
    python tools/decoder_fusion_ab.py --family qwen3 --out /tmp/r07_qwen3_raw.json
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

HID, NQ, NKV, HD = 4096, 32, 8, 128                  # shared by LLaMA-3-8B, Mistral-7B and Qwen3-8B
LLAMA3_8B = dict(vocab_size=128256, hidden_size=HID, intermediate_size=14336, num_hidden_layers=32,
                 num_attention_heads=NQ, num_key_value_heads=NKV, max_position_embeddings=8192, rms_norm_eps=1e-5,
                 rope_theta=500000.0, attn_implementation="sdpa")
MISTRAL_7B = dict(vocab_size=32768, hidden_size=HID, intermediate_size=14336, num_hidden_layers=32,
                  num_attention_heads=NQ, num_key_value_heads=NKV, head_dim=HD, max_position_embeddings=8192,
                  rms_norm_eps=1e-5, rope_theta=1000000.0, sliding_window=None, attn_implementation="sdpa")
QWEN3_8B = dict(vocab_size=151936, hidden_size=HID, intermediate_size=12288, num_hidden_layers=36,
                num_attention_heads=NQ, num_key_value_heads=NKV, head_dim=HD, max_position_embeddings=8192,
                rms_norm_eps=1e-6, rope_theta=1000000.0, attn_implementation="sdpa")
FAMILIES = {"llama": ("Llama", LLAMA3_8B), "mistral": ("Mistral", MISTRAL_7B), "qwen3": ("Qwen3", QWEN3_8B)}


def kernel_bytes(T: int, cfg: dict = LLAMA3_8B, qk_norm: bool = False) -> dict:
    """Bytes each kernel must move at least (bf16 tensors, fp32 rstd; weights and cos/sin tables are negligible)."""
    row, q_k = 2 * T * HID, 2 * T * (NQ + NKV) * HD
    mlp = 2 * T * cfg["intermediate_size"]
    out = {"rmsnorm_fwd": 2 * row + 4 * T,                      # x -> y, rstd
           "add_rmsnorm_fwd": 4 * row + 4 * T,                  # res, a -> h, y, rstd
           "rmsnorm_bwd_dres": 4 * row + 4 * T,                 # x, dy, dres, rstd -> dx
           "rope_fwd": 2 * q_k,                                 # q, k -> q, k
           "rope_bwd": 2 * q_k,
           "swiglu_fwd": 3 * mlp,                               # g, u -> h
           "swiglu_bwd": 5 * mlp}                               # g, u, dh -> dg, du
    if qk_norm:
        rows = T * (NQ + NKV)
        out["qk_norm_rope_fwd"] = 2 * q_k + 4 * rows            # q, k -> q, k, rstd
        out["qk_norm_rope_bwd"] = 3 * q_k + 4 * rows            # q, k, dq_out, dk_out, rstd -> dq, dk
    return out


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


def per_kernel(T, iters, hbm_gbs, family="llama"):
    import importlib

    import torch
    from sparse_matrix_tuning_b200 import ops
    _, cfg = FAMILIES[family]
    apply_rotary_pos_emb = importlib.import_module(f"transformers.models.{family}.modeling_{family}").apply_rotary_pos_emb
    INTER = cfg["intermediate_size"]
    dev, eps = "cuda", cfg["rms_norm_eps"]
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
    pos = torch.arange(S, device=dev).float()[:, None] * (cfg["rope_theta"] ** (-torch.arange(0, HD, 2, device=dev) / HD))
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
    composed = {}
    if family == "qwen3":
        wq = (1 + 0.1 * torch.randn(HD, device=dev)).bfloat16()
        wk = (1 + 0.1 * torch.randn(HD, device=dev)).bfloat16()

        def hf_head_norm(t, wt):
            tf = t.float()
            return wt * (tf * torch.rsqrt(tf.pow(2).mean(-1, keepdim=True) + eps)).to(t.dtype)

        def composed_fwd():                       # existing kernels: one norm launch per tensor, then RoPE
            yq = ops.rmsnorm_forward(q, wq, eps)[0]
            yk = ops.rmsnorm_forward(k, wk, eps)[0]
            return ops.rope_forward(yq, yk, cos, sin)

        _qo, _ko, rstd_q, rstd_k = ops.qk_norm_rope_forward(q, k, wq, wk, eps, eps, cos, sin)
        _yq, rq_rows, _ = ops.rmsnorm_forward(q, wq, eps)
        _yk, rk_rows, _ = ops.rmsnorm_forward(k, wk, eps)

        def composed_bwd():
            dq_n, dk_n = ops.rope_backward(dq_o, dk_o, cos, sin)
            return ops.rmsnorm_backward(q, wq, rq_rows, dq_n), ops.rmsnorm_backward(k, wk, rk_rows, dk_n)

        qn, kn = q.clone().requires_grad_(True), k.clone().requires_grad_(True)
        rqh, rkh = apply_rotary_pos_emb(hf_head_norm(qn, wq).transpose(1, 2), hf_head_norm(kn, wk).transpose(1, 2),
                                        cos, sin)
        cases["qk_norm_rope_fwd"] = (
            lambda: ops.qk_norm_rope_forward(q, k, wq, wk, eps, eps, cos, sin),
            lambda: apply_rotary_pos_emb(hf_head_norm(q, wq).transpose(1, 2), hf_head_norm(k, wk).transpose(1, 2),
                                         cos, sin))
        cases["qk_norm_rope_bwd"] = (
            lambda: ops.qk_norm_rope_backward(q, k, wq, wk, rstd_q, rstd_k, cos, sin, dq_o, dk_o),
            lambda: torch.autograd.grad((rqh, rkh), (qn, kn), (dq_o.transpose(1, 2), dk_o.transpose(1, 2)),
                                        retain_graph=True))
        composed = {"qk_norm_rope_fwd": composed_fwd, "qk_norm_rope_bwd": composed_bwd}
    nbytes = kernel_bytes(T, cfg, qk_norm=family == "qwen3")
    out = {}
    for name, (ours, hf) in cases.items():
        t_ours, t_hf = time_ms(ours, iters, flush), time_ms(hf, iters, flush)
        gbs = nbytes[name] / (t_ours * 1e-3) / 1e9
        out[name] = {"us": t_ours * 1e3, "hf_us": t_hf * 1e3, "speedup_vs_hf": t_hf / t_ours, "bytes": nbytes[name],
                     "gb_per_s": gbs, "fraction_of_hbm_peak": gbs / hbm_gbs}
        if name in composed:
            t_c = time_ms(composed[name], iters, flush)
            out[name].update(existing_kernels_us=t_c * 1e3, speedup_vs_existing_kernels=t_c / t_ours)
    return out


def one_layer(T, iters, family="llama"):
    """One decoder layer, fwd + recompute + bwd (non-reentrant checkpoint), elementwise fusion on / off."""
    import importlib

    import torch
    import transformers
    from torch.utils.checkpoint import checkpoint
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.smt import smt as M
    prefix, fam_cfg = FAMILIES[family]
    mod = importlib.import_module(f"transformers.models.{family}.modeling_{family}")
    cfg = getattr(transformers, prefix + "Config")(**{**fam_cfg, "num_hidden_layers": 1})
    torch.manual_seed(0)
    torch.set_default_dtype(torch.bfloat16)
    try:
        layer = getattr(mod, prefix + "DecoderLayer")(cfg, 0).cuda()
    finally:
        torch.set_default_dtype(torch.float32)
    for p in layer.parameters():
        p.requires_grad_(False)
    S = 512
    B = T // S
    x = torch.randn(B, S, HID, device="cuda").bfloat16().requires_grad_(True)
    dout = torch.randn(B, S, HID, device="cuda").bfloat16()
    pos = torch.arange(S, device="cuda")[None]
    pe = getattr(mod, prefix + "RotaryEmbedding")(cfg).cuda()(x, pos)

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


def whole_step(steps, reps, batch, seq, family="llama"):
    """The SMT step of bench.py at its default shape: fusion on / off alternating, q/k/v fused in both.  LLaMA: arms
    `fused` / `unfused` differ in the elementwise ops; other families: `fused` adds the fused causal-LM loss, `unfused`
    is what these models got before (q/k/v GEMMs fused, everything else transformers')."""
    import random

    import torch
    import transformers
    from sparse_matrix_tuning_b200 import decoder_fusion as D
    from sparse_matrix_tuning_b200.optim import SMTAdam
    from sparse_matrix_tuning_b200.smt import smt as M
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    prefix, fam_cfg = FAMILIES[family]
    cfg = getattr(transformers, prefix + "Config")(**fam_cfg)
    torch.manual_seed(1234)
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device("cuda"):
            model = getattr(transformers, prefix + "ForCausalLM")(cfg)
    finally:
        torch.set_default_dtype(torch.float32)
    model.config.use_cache = False
    # q/k/v blocks as bench.py's gradient-based selection picks at its default ratio (LLaMA-3-8B: 869), at random
    n_blocks = 869 if family == "llama" else H.block_budget(model, 0.0071)
    layers = cfg.num_hidden_layers
    rng = random.Random(0)
    sel = {}
    shapes = {"q_proj": (HID // 256, HID // 256), "k_proj": (NKV * HD // 256, HID // 256),
              "v_proj": (NKV * HD // 256, HID // 256)}
    cand = [(kind, l, r, c) for l in range(layers) for kind, (R, C) in shapes.items() for r in range(R)
            for c in range(C)]
    for kind, l, r, c in sorted(rng.sample(cand, n_blocks)):
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
    peak = {"fused": [], "unfused": []}
    for _ in range(reps):
        for arm in ("fused", "unfused"):
            M.fuse_qkv_projections(model)
            if arm == "unfused":
                D.remove_all(model)
            elif family != "llama":
                M.fuse_causal_lm_loss(model)
            for i in range(2):
                step(ids[i])
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for t in ids:
                step(t)
            b.record()
            torch.cuda.synchronize()
            res[arm].append(a.elapsed_time(b) / steps)
            peak[arm].append(torch.cuda.max_memory_allocated())
            M.unfuse_qkv_projections(model)
            M.unfuse_causal_lm_loss(model)
    M.set_grouped_backward(False)
    out = {"ms_per_step": res, "steps_per_rep": steps, "reps": reps, "tokens_per_step": batch * seq,
           "speedup_min_over_pairs": min(u / f for u, f in zip(res["unfused"], res["fused"]))}
    if family != "llama":
        out.update(family=family, layers=layers, qkv_blocks=n_blocks, max_memory_allocated_bytes=peak,
                   tokens_per_s={arm: [batch * seq / (ms * 1e-3) for ms in v] for arm, v in res.items()},
                   fused_faster_in_every_pair=all(f < u for f, u in zip(res["fused"], res["unfused"])))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--family", choices=sorted(FAMILIES), default="llama")
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
        info = {"tokens": args.tokens,
                "bytes": kernel_bytes(args.tokens, FAMILIES[args.family][1], qk_norm=args.family == "qwen3")}
        if args.family != "llama":
            info["family"] = args.family
        print(json.dumps(info))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    t0 = time.time()
    result = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "tokens": args.tokens,
              "hbm_gbs_reference": args.hbm_gbs, "l2_flush_bytes_between_launches": 256 << 20}
    if args.family != "llama":
        result["family"] = args.family
    result["per_kernel"] = per_kernel(args.tokens, args.iters, args.hbm_gbs, args.family)
    torch.cuda.empty_cache()
    result["one_layer_fwd_recompute_bwd"] = one_layer(args.tokens, args.layer_iters, args.family)
    torch.cuda.empty_cache()
    if not args.skip_step:
        result["whole_step"] = whole_step(args.steps, args.reps, 16, 512, args.family)
    result["wall_s"] = time.time() - t0
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
