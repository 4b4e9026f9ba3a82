#!/usr/bin/env python
"""bench.py — headline benchmark of the SMT hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own modules on the box's host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json metric "tokens/sec/GPU (LLaMA-3-8B SMT 0.71%)", configs[2]/[3]): a random-init LLaMA-3-8B
(`LlamaForCausalLM`, bf16) whose q/k/v projections own 869 selected 256x256 blocks (0.71 % of the 122 528 blocks the
reference's budget counts, fine_tune.py:231-239).  One STEP = forward + backward (the selected-block gradients come
from the tcgen05 block-gradient GEMM, flushed in GPU-filling chunks) + [N>1: all-reduce of the flat compact-gradient
buffer, chunk by chunk on a side stream while the backward pass continues] + one fused compact-Adam/clip/write-back
launch, on synthetic tokens (uniform ids, labels = ids).  Before the timed steps the script runs the warm-up part of
the path (capture-only: gradient-capture passes with grad-ready hooks feeding the on-device block-score accumulators,
block-score finalize, exact top-k, freeze, convert) and reports it separately.

One JSON line on stdout (rank 0).  `value` = tokens/s over all ranks with inputs resident in HBM; `e2e` = the same
step with the token ids copied from pinned host memory and the loss read back every step; `roofline` describes the
dominant SMT kernel (block-gradient GEMM) from CUDA-event timings taken live inside the timed region, `roofline.also`
the HBM-bound kernels (compact Adam in-step; score kernels warm, at the full LLaMA-3-8B q/k/v size) and four
BASELINE-config-2 sweep points; `cpu_baseline` times the reference's own modules (oracle/_ref, staged by
oracle/build_ref.py) on the host cores (bounded sample); `secondary_comparator` runs those same reference modules
eagerly on the B200 for full steps of the same workload; `dp_check` (N>1) verifies the data-parallel numerics;
`config5` re-runs the step with attention + MLP blocks (BASELINE configs[4] shape).
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LLAMA3_8B = dict(vocab_size=128256, hidden_size=4096, intermediate_size=14336, num_hidden_layers=32,
                 num_attention_heads=32, num_key_value_heads=8, max_position_embeddings=8192, rope_theta=500000.0,
                 rms_norm_eps=1e-5, tie_word_embeddings=False)
ATTN_RATIO = 0.0071       # "SMT 0.71 %": int(0.0071 * 122528) = 869 blocks  (BASELINE.md section 1)
CONFIG5_RATIO = 0.0043    # BASELINE configs[4] shape: 0.0043 attention + 0.0043 MLP -> 526 + 526 blocks (0.86 %)
BLOCK = 256
METRIC = "tokens/sec (LLaMA-3-8B SMT 0.71%), aggregate over n_gpus (per-GPU = value / n_gpus)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=16, help="sequences per GPU")
    ap.add_argument("--seq", type=int, default=512)
    ap.add_argument("--layers", type=int, default=32, help="(debug only) fewer layers => config.workload says so")
    ap.add_argument("--no-ckpt", action="store_true", help="disable gradient checkpointing (reference: on, fine_tune.py:192)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seq", type=int, default=512, help="tokens of the bounded CPU sample")
    ap.add_argument("--attn-ratio", type=float, default=ATTN_RATIO, help="fine_tune.py --downsample_attention_blocks_ratio")
    ap.add_argument("--mlp-ratio", type=float, default=0.0, help="fine_tune.py --downsample_mlp_blocks_ratio (0 = off)")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra records (no-checkpointing, config 5, "
                                                            "config-2 points, score kernels, eager reference)")
    ap.add_argument("--no-group", action="store_true", help="launch the block-gradient GEMM per module instead of grouped")
    ap.add_argument("--no-fuse-qkv", action="store_true", help="keep one library GEMM per q/k/v module instead of the fused "
                                                               "tcgen05 projection / input-gradient kernels")
    ap.add_argument("--no-overlap", action="store_true", help="N>1: one blocking all-reduce after backward (round-1 behaviour)")
    ap.add_argument("--chunk-blocks", type=int, default=192, help="grouped GEMM flush granularity during backward (N>1)")
    ap.add_argument("--capture-steps", type=int, default=4, help="gradient-capture passes of the warm-up phase")
    ap.add_argument("--torch-profile", type=str, default="", help="(diagnostic) write a torch.profiler kernel table of two "
                                                                  "steps to this file: GPU busy time vs step time")
    ap.add_argument("--dump-outputs", type=str, default="", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (see "
                         "dump_outputs) so that two builds can be compared output for output; the warm-up then "
                         "runs its attention backward on the deterministic math kernel, so its reported times are "
                         "those of that kernel and it may select other blocks than a run without this flag")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi sampled every 200 ms while the timed region runs (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                                  ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own modules (oracle/_ref, else the oracle port) on the host cores
# ---------------------------------------------------------------------------------------------------------------

def _reference_modules():
    """(LinearLayer_MatrixSparsity class of the reference, kind).  The reference is pure Python: oracle/build_ref.py
    stages its two modules under oracle/_ref/ and oracle/ref_shim.py imports them unmodified (fake `deepspeed`)."""
    try:
        from oracle import ref_shim
        if ref_shim.reference_available():
            ref_smt, _ref_helper = ref_shim.load_reference()
            return ref_smt, "reference"
    except Exception as e:  # pragma: no cover - staged copy missing / import problem: fall back to the port
        sys.stderr.write(f"[bench] reference modules unavailable ({type(e).__name__}: {e}); using the oracle port\n")
    return None, "port"


def cpu_reference_arm(steps: int, warmup: int, seq: int):
    """Bounded sample: ONE LLaMA-3-8B decoder layer (of 32) in bf16 on the host cores, q/k/v converted to the
    REFERENCE's `LinearLayer_MatrixSparsity` (27 = round(869/32) selected 256x256 blocks), batch 1 x `seq` tokens:
    forward (with the per-forward scatter loop), backward (per-block bmm + sum + copy loop, smt.py:386-404) and a clipped
    AdamW step on the compact parameters.  Returns the MEASURED per-layer step time; tokens/s for the whole model is an
    extrapolation, seq / (32 * t_layer): embeddings, final norm, lm_head and the loss are left out, which favours the
    CPU arm."""
    import torch
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer, LlamaRotaryEmbedding

    ref_smt, kind = _reference_modules()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(1234)
    cfg = LlamaConfig(**{**LLAMA3_8B, "num_hidden_layers": 1}, attn_implementation="sdpa")
    layer = LlamaDecoderLayer(cfg, layer_idx=0).to(torch.bfloat16)
    rope = LlamaRotaryEmbedding(cfg)
    for p in layer.parameters():
        p.requires_grad = False
    g = torch.Generator().manual_seed(7)
    per_module = {"q_proj": 15, "k_proj": 6, "v_proj": 6}            # 27 blocks/layer, k/v (GQA) are 4 x 16 blocks
    sparse = []
    for name, n in per_module.items():
        lin = getattr(layer.self_attn, name)
        rows, cols = lin.weight.shape[0] // BLOCK, lin.weight.shape[1] // BLOCK
        perm = torch.randperm(rows * cols, generator=g)[:n]
        idx = [(int(p) // cols, int(p) % cols) for p in perm]
        if ref_smt is not None:
            mod = ref_smt.LinearLayer_MatrixSparsity(lin.weight, bias=None, index_list=idx)   # smt.py:302 (unmodified)
        else:
            from oracle import smt_oracle as O
            mod = O.OracleSparseLinear(lin.weight, idx, BLOCK)
        setattr(layer.self_attn, name, mod)
        sparse.append(mod)
    params = [m.selected_weight for m in sparse]
    opt = torch.optim.AdamW(params, lr=1e-4, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.0)
    x = torch.randn(1, seq, cfg.hidden_size, generator=g).to(torch.bfloat16).requires_grad_(True)
    pos = torch.arange(seq).unsqueeze(0)
    cos_sin = rope(x, pos)

    def one_step():
        opt.zero_grad()
        out = layer(x, position_embeddings=cos_sin, position_ids=pos, attention_mask=None)
        out = out[0] if isinstance(out, tuple) else out
        out.float().pow(2).mean().backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()

    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    tokens_per_s = seq / (dt * LLAMA3_8B["num_hidden_layers"])
    what = ("the reference's own LinearLayer_MatrixSparsity / linearZ (oracle/_ref, unmodified smt.py)" if kind == "reference"
            else "oracle port of smt.py forward/backward (oracle/_ref not staged)")
    sample = (f"1 of 32 LLaMA-3-8B decoder layers, bf16, batch 1 x {seq} tokens, 27 q/k/v blocks, {what} + clipped AdamW; "
              f"measured {dt * 1e3:.1f} ms per layer-step; tokens/s = {seq}/(32*t_layer) is an extrapolation; "
              f"{steps} steps after {warmup} warm-up")
    return tokens_per_s, dt * 1e3, cores, sample, kind


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tps, ms, cores, sample, kind = cpu_reference_arm(args.steps, args.warmup, args.cpu_seq)
    line = {"impl": "reference", "metric": METRIC, "value": tps, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms,                                   # MEASURED: one decoder layer, batch 1 x cpu_seq tokens
            "extrapolated_full_model_ms_per_step": ms * LLAMA3_8B["num_hidden_layers"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"LLaMA-3-8B SMT 0.71% q/k/v gradient-based selection, bf16, seq {args.seq} x batch "
                                   f"{args.batch} per GPU",
                       "note": "same workload as the GPU arm, measured on a bounded sample (see cpu_baseline.sample): a step "
                               "here is ONE decoder layer at batch 1; `value` extrapolates it to the 32-layer model"},
            "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------

def build_model(args, device):
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(**{**LLAMA3_8B, "num_hidden_layers": args.layers}, attn_implementation="sdpa")
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(device):
            model = LlamaForCausalLM(cfg)
    finally:
        torch.set_default_dtype(torch.float32)
    model.config.use_cache = False
    return model


DUMP_SAMPLE = 1 << 22       # positions kept per weight array: 2 x 16 MB of float32


def dump_outputs(out_dir, loss, model, opt):
    """What the last timed step hands its caller: `loss.npy` (float64, [1]; this rank's loss on its own micro-batch,
    not the mean over data-parallel ranks) and the trainable compact weights it
    updated, as the model holds them (`selected_weight.npy`, bf16 values in float32) and as the optimizer's fp32
    masters (`master_weight.npy`).  Both are the concatenation of every trainable parameter in `named_parameters()`
    order, reduced to the same fixed, seeded sample of at most DUMP_SAMPLE sorted positions."""
    import numpy as np
    import torch
    params = [p for _n, p in model.named_parameters() if p.requires_grad]
    weights = torch.cat([p.detach().reshape(-1).float() for p in params])
    masters = torch.cat([opt.state[p]["master"].reshape(-1) for p in params])
    if weights.numel() > DUMP_SAMPLE:
        pos = torch.randint(0, weights.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).unique()
        pos = pos.to(weights.device)
        weights, masters = weights[pos], masters[pos]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss.item()], dtype=np.float64))
    np.save(os.path.join(out_dir, "selected_weight.npy"), weights.cpu().numpy())
    np.save(os.path.join(out_dir, "master_weight.npy"), masters.cpu().numpy())


def _median_ms(fn, iters=5, warmup=2, flush=None):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def score_kernel_rooflines(device, hbm_peak):
    """The three warm-up scoring kernels at the full LLaMA-3-8B q/k/v size (805 306 368 elements = one step's captured
    gradients), warm, CUDA events; operands are 1.6-3.2 GB, far larger than L2."""
    import torch
    from sparse_matrix_tuning_b200 import ops
    R, C = 16384, 49152                                            # 805 306 368 elements
    n = R * C
    grad = torch.empty(R, C, dtype=torch.bfloat16, device=device).normal_()
    acc = torch.zeros(R, C, dtype=torch.float32, device=device)
    sums = torch.zeros(R // BLOCK, C // BLOCK, dtype=torch.float32, device=device)
    out = {}
    for name, fn, bpe in (("score_accumulate", lambda: ops.score_accumulate(acc, grad), 10),
                          ("block_score_reduce", lambda: ops.block_score_reduce(acc, BLOCK, "mean_abs"), 4),
                          ("block_sum_accumulate", lambda: ops.block_sum_accumulate(sums, grad, BLOCK), 2)):
        ms = _median_ms(fn)
        gbs = n * bpe / (ms * 1e-3) / 1e9
        out[name] = {"bound": "hbm", "elements": n, "bytes_per_elem": bpe, "avg_ms": ms, "achieved_gbs": gbs,
                     "peak_gbs": hbm_peak, "frac": gbs / hbm_peak}
    del grad, acc, sums
    torch.cuda.empty_cache()
    return out


def config2_points(device, peaks):
    """Four BASELINE configs[1] sweep points (per-module launches, the regime the zero-edit DeepSpeed drop-in runs in):
    CUDA events, 256 MB memset between iterations (2x L2).  frac = max(flops/bf16 burst peak, min HBM bytes/HBM peak) /
    measured time, the same definition as tools/kernel_sweep.py."""
    import torch
    from sparse_matrix_tuning_b200 import ops
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    peak_tf, hbm = peaks.get("bf16_tflops", 1599.5), peaks.get("hbm_gbs", 6545.6)
    g = torch.Generator().manual_seed(0)
    pts = []
    for label, fout, fin, b, frac_sel, T, pattern in (
            ("q 4096x4096", 4096, 4096, 256, 0.05, 16384, "random"),
            ("gate/up 14336x4096", 14336, 4096, 256, 0.05, 8192, "random"),
            ("q 4096x4096", 4096, 4096, 128, 0.05, 16384, "random"),
            ("q 4096x4096", 4096, 4096, 64, 0.05, 16384, "clustered")):
        rows, cols = fout // b, fin // b
        n = max(1, int(frac_sel * rows * cols))
        if pattern == "random":
            perm = torch.randperm(rows * cols, generator=g)[:n]
            idx = [(int(p) // cols, int(p) % cols) for p in perm]
        else:                                                      # whole block rows, then a partial one
            idx = [(i // cols, i % cols) for i in range(n)]
        x = torch.randn(T, fin, device=device).bfloat16()
        dy = torch.randn(T, fout, device=device).bfloat16()
        rc = ops.make_block_rc(idx, device)
        out = torch.empty(n * b, b, dtype=torch.bfloat16, device=device)
        ms = _median_ms(lambda: ops.block_grad_gemm(x, dy, rc, b, out=out, index_list=idx), iters=7, flush=flush)
        flops = 2.0 * b * b * T * n
        min_bytes = 2.0 * T * b * (len({r for r, _ in idx}) + len({c for _, c in idx})) + 2.0 * n * b * b
        bound_s = max(flops / (peak_tf * 1e12), min_bytes / (hbm * 1e9))
        pts.append({"weight": label, "block": b, "sparsity": frac_sel, "pattern": pattern, "T": T, "n_blocks": n,
                    "kernel": ops.LAST_SINGLE.get("kernel"),
                    "us": ms * 1e3, "tflops": flops / (ms * 1e-3) / 1e12,
                    "bound": "tensor" if flops / (peak_tf * 1e12) >= min_bytes / (hbm * 1e9) else "hbm",
                    "frac_of_roofline": bound_s / (ms * 1e-3), "frac_of_bf16_burst": flops / (ms * 1e-3) / 1e12 / peak_tf})
        del x, dy, out
    del flush
    torch.cuda.empty_cache()
    return pts


def fused_qkv_ab(device, T, peaks):
    """f-2, driver-visible A/B on this box: the fused tcgen05 q/k/v projection and the fused input gradient against the
    library GEMMs they replace (three `torch.matmul` per direction + the two adds autograd inserts between the three
    input gradients), LLaMA-3-8B q/k/v shapes at this run's token count.  CUDA events, 256 MB memset between
    iterations."""
    import torch
    from sparse_matrix_tuning_b200 import ops
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    K, Ns = 4096, [4096, 1024, 1024]
    x = torch.randn(T, K, device=device).bfloat16()
    ws = [(torch.randn(n, K, device=device) * 0.02).bfloat16() for n in Ns]
    dys = [torch.randn(T, n, device=device).bfloat16() for n in Ns]
    flops = 2.0 * T * K * sum(Ns)
    peak = peaks.get("bf16_tflops", 1599.5)

    def lib_dgrad():
        acc = torch.matmul(dys[0], ws[0])
        for dy, w in zip(dys[1:], ws[1:]):
            acc = acc + torch.matmul(dy, w)
        return acc

    out = {"shape": f"x[{T}, {K}] x [Wq; Wk; Wv]^T -> {'+'.join(map(str, Ns))} columns; dx over K = {sum(Ns)}",
           "kernel": "fused_dense_umma_2sm_kernel (persistent, cta_group::2, 256x256 tiles, 6 stages, 2 TMEM accumulators)"}
    for name, lib_fn, fused_fn in (("forward", lambda: [torch.matmul(x, w.t()) for w in ws],
                                    lambda: ops.fused_linear_forward(x, ws)),
                                   ("dgrad", lib_dgrad, lambda: ops.fused_linear_dgrad(dys, ws))):
        t_lib = _median_ms(lib_fn, iters=9, warmup=3, flush=flush)
        t_fus = _median_ms(fused_fn, iters=9, warmup=3, flush=flush)
        out[name] = {"library_us": t_lib * 1e3, "library_tflops": flops / (t_lib * 1e-3) / 1e12,
                     "fused_us": t_fus * 1e3, "fused_tflops": flops / (t_fus * 1e-3) / 1e12,
                     "speedup": t_lib / t_fus, "bound": "tensor", "frac_of_bf16_burst": flops / (t_fus * 1e-3) / 1e12 / peak}
    lib_total = 2 * out["forward"]["library_us"] + out["dgrad"]["library_us"]
    fus_total = 2 * out["forward"]["fused_us"] + out["dgrad"]["fused_us"]
    out["per_layer_step_us"] = {"library": lib_total, "fused": fus_total, "speedup": lib_total / fus_total,
                                "note": "forward x 2 (gradient checkpointing recomputes it) + input gradient"}
    del flush
    torch.cuda.empty_cache()
    return out


def full_ft_warmup_record(model, dev_ids, steps=2):
    """The reference's warm-up policy on ONE B200: real full-fine-tuning steps (every parameter trainable, AdamW betas
    (0.9, 0.95), clip 1.0 - fine_tune.py:168-190, 773) while the q/k/v gradients are captured at grad-ready time
    (fine_tune.py:716-768).  The reference needs ZeRO + CPU offload for this at 8 B; 180 GB of HBM hold bf16 parameters,
    bf16 gradients and the (bf16) Adam moments with room to spare, so it simply runs.  Reports step time and peak memory;
    the bench keeps capture-only as its default warm-up because it leaves the weights untouched and costs a third less."""
    import torch
    from sparse_matrix_tuning_b200.warmup import WarmupGradAccumulator
    try:
        for p in model.parameters():
            p.requires_grad = True
        params = [p for p in model.parameters()]
        opt = torch.optim.AdamW(params, lr=9.65e-6, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.0, fused=True)
        acc = WarmupGradAccumulator(block=BLOCK, mode="block_sum", mlp=False, attention=True)
        acc.attach(model, free_grads=False)                       # the optimizer still needs the gradients
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        times = []
        for i in range(steps):
            t0 = time.perf_counter()
            ids = dev_ids[-1 - (i % 2)]
            loss = model(input_ids=ids, labels=ids, use_cache=False).loss
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
            opt.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) * 1e3)
        acc.detach()
        peak = torch.cuda.max_memory_allocated()
        del opt, params
        model.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
        return {"what": "real full-FT warm-up steps with on-device capture (the reference's policy, fine_tune.py:168-190, "
                        "716-773) on one B200: all 8.03 B parameters trainable, torch fused AdamW (bf16 moments), clip 1.0",
                "steps": steps, "ms_per_step": times, "peak_memory_gb": peak / 1e9, "loss_last": loss.item(), "_acc": acc}
    except Exception as e:
        torch.cuda.empty_cache()
        return {"error": f"{type(e).__name__}: {e}"}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from sparse_matrix_tuning_b200 import _lib, dp, ops
    from sparse_matrix_tuning_b200.optim import SMTAdam
    from sparse_matrix_tuning_b200.smt import smt as M, smt_helper as H
    from sparse_matrix_tuning_b200.warmup import WarmupGradAccumulator

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    _lib.load()                                                   # fail loudly if the extension is missing
    peaks = load_peaks()
    hbm_peak = peaks.get("hbm_gbs", 6650.0)

    torch.manual_seed(1234)                                       # identical weights on every rank
    model = build_model(args, device)
    vocab = LLAMA3_8B["vocab_size"]
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)  # per-rank data (weak scaling)
    B, S = args.batch, args.seq
    T = B * S
    n_batches = args.warmup + args.steps + 2
    host_ids = [torch.randint(0, vocab, (B, S), generator=gen).pin_memory() for _ in range(n_batches)]
    dev_ids = [t.to(device) for t in host_ids]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up part of the path (timed separately) ---------------------------------------------------------------
    # Policy (SURVEY 8f-3, declared): CAPTURE-ONLY.  The reference runs `--full_ft_steps` real full-fine-tuning steps
    # while it captures (fine_tune.py:168-190, 716-773), which for 8 B parameters needs ZeRO + CPU offload (16 GB bf16
    # + 96 GB fp32 Adam state + gradients).  Here the warm-up runs K gradient-capture passes WITHOUT optimizer steps:
    # grad-ready hooks feed every q/k/v (and MLP) gradient to the on-device block-sum accumulators the moment autograd
    # has produced it and release it, so the pass never holds more than one targeted gradient.
    dims = H.targeted_module_dims(model)                          # fine_tune.py:221-228
    total_blocks = H.num_total_blocks(model, BLOCK)               # fine_tune.py:231-234
    n_attn = H.block_budget(model, args.attn_ratio, BLOCK)        # fine_tune.py:236
    n_mlp = H.block_budget(model, args.mlp_ratio, BLOCK) if args.mlp_ratio > 0 else 0   # fine_tune.py:239

    def set_capture_requires_grad(with_mlp):
        for name, p in model.named_parameters():
            p.requires_grad = (("self_attn" in name) and any(k in name for k in ("q_proj", "k_proj", "v_proj"))) or \
                              (with_mlp and "mlp" in name)

    set_capture_requires_grad(n_mlp > 0)
    if not args.no_ckpt:
        # non-reentrant checkpointing keeps the whole backward in ONE autograd graph task, so the block-gradient GEMMs
        # of all modules can be deferred to grouped launches
        model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
        model.enable_input_require_grads()
    model.train()

    def capture_phase(with_mlp, steps):
        """`steps` capture passes with grad-ready hooks; returns (attention acc, mlp acc, per-pass ms list)."""
        # two accumulators, as the driver keeps `attention_warmup_grads` and `warmup_grads` apart (fine_tune.py:723-765)
        acc_a = WarmupGradAccumulator(block=BLOCK, mode="block_sum", mlp=False, attention=True)
        acc_m = WarmupGradAccumulator(block=BLOCK, mode="block_sum", mlp=True, attention=False) if with_mlp else None
        acc_a.attach(model, free_grads=True)
        if acc_m is not None:
            acc_m.attach(model, free_grads=True)
        times = []
        for i in range(steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ids = dev_ids[-1 - (i % 2)]
            model(input_ids=ids, labels=ids, use_cache=False).loss.backward()
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) * 1e3)
        acc_a.detach()
        if acc_m is not None:
            acc_m.detach()
        model.zero_grad(set_to_none=True)
        dp.allreduce_block_sums(acc_a)                            # scores of the DP-mean gradient on every rank
        if acc_m is not None:
            dp.allreduce_block_sums(acc_m)
        return acc_a, acc_m, times

    # With --dump-outputs the warm-up's backward passes, which decide the blocks the timed steps train, run on the math
    # attention kernel: the fused attention backward kernels accumulate in a run-dependent order, and the block scores
    # of a random-init model are near-ties, so otherwise two runs select different blocks.  The timed steps are unchanged.
    if args.dump_outputs:
        from torch.nn.attention import SDPBackend, sdpa_kernel
        warmup_attention = lambda: sdpa_kernel(SDPBackend.MATH)     # noqa: E731
    else:
        warmup_attention = contextlib.nullcontext

    # ---- extra (1 GPU): the reference's OWN warm-up policy - real full-fine-tuning steps while capturing ------------------
    full_ft = None
    if not args.no_extra and world == 1 and args.layers == 32:
        with warmup_attention():
            full_ft = full_ft_warmup_record(model, dev_ids, steps=2)
        set_capture_requires_grad(n_mlp > 0)
    launches_capture0 = ops.LAUNCHES["total"]
    with warmup_attention():
        acc, acc_mlp, capture_ms = capture_phase(n_mlp > 0, max(1, args.capture_steps))
    capture_launches = ops.LAUNCHES["total"] - launches_capture0
    # the same pass without any capture hooks: what the hooks + score kernels add per step
    plain_ms = None
    if not args.no_extra:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model(input_ids=dev_ids[-1], labels=dev_ids[-1], use_cache=False).loss.backward()
        torch.cuda.synchronize()
        plain_ms = (time.perf_counter() - t0) * 1e3
        model.zero_grad(set_to_none=True)

    def select(acc_a, acc_m, k_attn, k_mlp):
        keys, scores = acc_a.scores("mean_abs")
        s_attn = H.select_submatrix_from_scores(keys, scores, k_attn, "no_restriction")     # fine_tune.py:306-313
        s_mlp = {}
        if acc_m is not None and k_mlp > 0:
            keys_m, scores_m = acc_m.scores("mean_abs")
            s_mlp = H.select_submatrix_from_scores(keys_m, scores_m, k_mlp, "no_restriction")   # fine_tune.py:319-327
        dp.assert_same_selection(s_attn)
        dp.assert_same_selection(s_mlp)
        return s_attn, s_mlp

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sel_attn, sel_mlp = select(acc, acc_mlp, n_attn, n_mlp)
    torch.cuda.synchronize()
    t_select = time.perf_counter() - t0
    if full_ft is not None and "error" not in full_ft:
        # how much does the cheap capture-only policy change WHAT is selected?  (different batches and step counts too)
        acc_ft = full_ft.pop("_acc")
        keys_f, scores_f = acc_ft.scores("mean_abs")
        sel_f = H.select_submatrix_from_scores(keys_f, scores_f, n_attn, "no_restriction")
        a = {(k, rc) for k, v in sel_attn.items() for rc in v}
        bset = {(k, rc) for k, v in sel_f.items() for rc in v}
        full_ft["selection_overlap_with_capture_only"] = len(a & bset) / max(len(a | bset), 1)
        del acc_ft
    del acc, acc_mlp

    # ---- extra, before the model is converted: score-kernel rooflines and config-2 points (rank 0 only) -------------
    score_roof, cfg2, qkv_ab = None, None, None
    if not args.no_extra and rank == 0:
        def guarded(fn, *a):                                      # an extra record must never cost the headline
            try:
                return fn(*a)
            except Exception as e:
                torch.cuda.empty_cache()
                return {"error": f"{type(e).__name__}: {e}"}
        score_roof = guarded(score_kernel_rooflines, device, hbm_peak)
        cfg2 = guarded(config2_points, device, peaks)
        qkv_ab = guarded(fused_qkv_ab, device, T, peaks)
    barrier()

    def convert(s_attn, s_mlp):
        M.freeze_unselected_matrix_layer(model, s_mlp, s_attn)
        M.convert_linear_layer_to_matrix_sparsity(model, s_mlp, s_attn)
        groups = M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-4)
        return SMTAdam(groups, lr=1e-4, betas=(0.9, 0.95), max_grad_norm=1.0)

    opt = convert(sel_attn, sel_mlp)
    n_fused_layers = 0 if args.no_fuse_qkv else M.fuse_qkv_projections(model)
    sel = {**sel_attn, **sel_mlp}
    n_blocks = sum(len(v) for v in sel.values())
    trainable = opt.trainable_elements()
    overlap = world > 1 and not args.no_overlap and not args.no_group
    M.set_grouped_backward(not args.no_group, chunk_blocks=args.chunk_blocks if overlap else 0)
    exchange = dp.OverlappedGradExchange(opt) if overlap else None
    torch.cuda.empty_cache()

    phase_events = []                                             # per step: CUDA events at the phase boundaries

    def step(ids, record=False):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)] if record else None
        if record:
            ev[0].record()
        out = model(input_ids=ids, labels=ids, use_cache=False)
        if record:
            ev[1].record()
        out.loss.backward()
        if record:
            ev[2].record()
        if exchange is not None:
            exchange.finish()
        else:
            works = dp.allreduce_compact_grads(opt, async_op=True)
            for w in works:
                w.wait()
        if record:
            ev[3].record()
        opt.step()
        opt.zero_grad()
        if record:
            ev[4].record()
            phase_events.append(ev)
        return out.loss

    for i in range(args.warmup):
        step(dev_ids[i])

    # ---- data-parallel numerics check (N > 1): the N-rank exchange against single-process gradient accumulation ------
    dp_check = None
    if world > 1:
        ids_c = dev_ids[-2]
        snap = opt.snapshot()
        all_ids = [torch.empty_like(ids_c) for _ in range(world)]
        dist.all_gather(all_ids, ids_c)
        arena = opt._arenas[0]
        # (1) the data-parallel way: one micro-batch per rank, exchange, Adam.  The exchange keeps a copy of this rank's
        #     gradients as they were before each chunk was reduced, so the collective can be checked EXACTLY (same
        #     backward pass, no run-to-run noise): reduced buffer vs the fp32 sum of the gathered per-rank buffers.
        opt.zero_grad()
        local = torch.zeros_like(arena.flat_grad)
        if exchange is not None:
            exchange.keep_local = local
        model(input_ids=ids_c, labels=ids_c, use_cache=False).loss.backward()
        if exchange is not None:
            exchange.finish()
            exchange.keep_local = None
        else:
            M.flush_block_grads()
            local.copy_(arena.flat_grad)
            for w in dp.allreduce_compact_grads(opt, async_op=True):
                w.wait()
        dp_sum = arena.flat_grad.float().clone()
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local)
        exact = torch.zeros_like(dp_sum)
        for gth in gathered:
            exact += gth.float()
        del gathered, local
        ex_max = (dp_sum - exact).abs().max().item() / exact.abs().max().item()
        ex_l2 = ((dp_sum - exact).norm() / exact.norm()).item()
        del exact
        opt.step()
        master_dp = arena.master.clone()
        opt.restore(snap)
        # (2) single process: the same N micro-batches accumulated locally (sum), mean folded into grad_scale, no
        #     exchange; done twice to measure the run-to-run noise of the model's own backward pass (flash-attention
        #     backward accumulates with atomics), which bounds how close (1) and (2) can be
        if exchange is not None:
            exchange.active = False

        def accumulate_locally():
            opt.zero_grad()
            for ids in all_ids:
                model(input_ids=ids, labels=ids, use_cache=False).loss.backward()
            M.flush_block_grads()
            return arena.flat_grad.float().clone()

        ref_sum = accumulate_locally()
        opt.grad_scale = 1.0 / world
        opt.step()
        master_ref = arena.master.clone()
        opt.restore(snap)
        ref_sum2 = accumulate_locally()
        opt.zero_grad()
        if exchange is not None:
            exchange.active = True
        noise_l2 = ((ref_sum2 - ref_sum).norm() / ref_sum.norm()).item()
        del ref_sum2
        gmax = ref_sum.abs().max().item()
        grad_rel = (dp_sum - ref_sum).abs().max().item() / gmax
        grad_l2 = ((dp_sum - ref_sum).norm() / ref_sum.norm()).item()
        master_diff = (master_dp - master_ref).abs().max().item()
        lr = float(opt.param_groups[0]["lr"])
        # Tolerances.  Exchange vs exact fp32 sum of the per-rank bf16 buffers: NCCL adds N bf16 values with N - 1
        # roundings of <= 2^-8 relative each.  Exchange vs local accumulation: two DIFFERENT executions of the model's
        # backward pass (per-rank vs all on one GPU), so on top of the bf16 roundings of the two summation orders
        # ((2 N + 1) * 2^-8 worst case) they differ by that pass's own run-to-run noise, measured above.
        ex_tol = (world - 1) * 2.0 ** -8
        max_tol = (2 * world + 1) * 2.0 ** -8 + 8 * noise_l2
        l2_tol = 2.0 ** -7 + 3 * noise_l2
        dp_check = {"exchange_vs_exact_sum_max_rel": ex_max, "exchange_vs_exact_sum_rel_l2": ex_l2,
                    "exchange_tolerance_max_rel": ex_tol,
                    "grad_max_rel": grad_rel, "grad_max_tolerance": max_tol, "grad_rel_l2": grad_l2,
                    "grad_rel_l2_tolerance": l2_tol, "backward_rerun_noise_rel_l2": noise_l2,
                    "master_max_abs_diff": master_diff,
                    "master_tolerance": 2 * lr, "micro_batches": world,
                    "what": "(a) flat compact-gradient buffer after the N-rank exchange vs the fp32 sum of the gathered "
                            "per-rank buffers of the SAME backward pass; (b) the same buffer vs N micro-batches accumulated in "
                            "one process (fine_tune.py:712 semantics: mean over ranks, clip after the reduction), then one Adam "
                            "step from the same state; backward_rerun_noise = (b) repeated twice on one GPU"}
        t = torch.tensor([ex_max, ex_l2, grad_rel, grad_l2, master_diff, noise_l2], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dp_check["max_over_ranks"] = dict(zip(("exchange_vs_exact_sum_max_rel", "exchange_vs_exact_sum_rel_l2",
                                               "grad_max_rel", "grad_rel_l2", "master_max_abs_diff",
                                               "backward_rerun_noise_rel_l2"), t.tolist()))
        ok = ex_max <= ex_tol and ex_l2 <= 2.0 ** -8 and grad_rel <= max_tol and grad_l2 <= l2_tol and master_diff <= 2 * lr
        flag = torch.tensor([0.0 if ok else 1.0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        dp_check["passed"] = flag.item() == 0.0
        if not dp_check["passed"]:                                # reported in the JSON line; the measurement still runs
            sys.stderr.write(f"[bench] rank {rank}: data-parallel numerics check FAILED: {dp_check}\n")
        del dp_sum, ref_sum, master_dp, master_ref, snap

    # ---- timed region 1: inputs resident in HBM ------------------------------------------------------------------
    ops.enable_timing("block_grad_gemm")
    ops.enable_timing("compact_adam")
    ops.enable_timing("fused_linear_forward")
    ops.enable_timing("fused_linear_dgrad")
    if exchange is not None:
        exchange.profile = True
    launches0 = ops.LAUNCHES["total"]
    host0 = dict(ops.HOST_TIME)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = step(dev_ids[args.warmup + i], record=True)
    e1.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model, opt)
    ms_total = e0.elapsed_time(e1)
    launches = ops.LAUNCHES["total"] - launches0
    host_flush_ms = (ops.HOST_TIME["flush_s"] - host0["flush_s"]) * 1e3 / max(args.steps, 1)
    gemm_t = ops.collect_timing("block_grad_gemm")
    adam_t = ops.collect_timing("compact_adam")
    fwd_t = ops.collect_timing("fused_linear_forward")
    dgr_t = ops.collect_timing("fused_linear_dgrad")
    for name in ("block_grad_gemm", "compact_adam", "fused_linear_forward", "fused_linear_dgrad"):
        ops.enable_timing(name, False)
    grouped_shape = dict(ops.LAST_GROUP)
    sq_source = getattr(opt, "sqnorm_source", None)
    phases = [[ev[k].elapsed_time(ev[k + 1]) for k in range(4)] for ev in phase_events]
    phase_mean = [statistics.mean(p[k] for p in phases) for k in range(4)]
    exch_ms = None
    if exchange is not None:
        exchange.profile = False
        per_chunk = [a.elapsed_time(b) for a, b in exchange.events]
        exch_ms = {"chunks_per_step": len(per_chunk) / max(args.steps, 1),
                   "allreduce_plus_sqnorm_ms_per_step_on_side_stream": sum(per_chunk) / max(args.steps, 1),
                   "max_chunk_ms": max(per_chunk) if per_chunk else None}
        exchange.events = []
    # ---- timed region 2: end to end (pinned host ids in, loss value out, every step) ------------------------------
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    last = None
    for i in range(args.steps):
        ids = host_ids[args.warmup + i].to(device, non_blocking=True)
        last = step(ids).item()
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    params_identical = dp.replicas_identical(opt) if world > 1 else None
    if world > 1 and not params_identical:
        sys.stderr.write(f"[bench] rank {rank}: replicas DIVERGED: flat parameters / fp32 masters differ between ranks\n")
    if args.torch_profile and rank == 0:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            t0 = time.perf_counter()
            for i in range(2):
                step(dev_ids[args.warmup + i])
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
        ka = prof.key_averages()
        busy = sum(e.self_device_time_total for e in ka) / 1e3
        with open(args.torch_profile, "w") as f:
            f.write(f"two steps: wall {wall:.1f} ms (under the profiler), sum of device kernel time {busy:.1f} ms "
                    f"=> GPU busy {100 * busy / wall:.1f} %\n\n")
            f.write(ka.table(sort_by="device_time_total", row_limit=40))
    # ---- extra (reported, not the headline): the same step WITHOUT activation recomputation ------------------------
    ms_nockpt = None
    if not args.no_ckpt and not args.no_extra:
        model.gradient_checkpointing_disable()
        for i in range(2):
            step(dev_ids[i])
        barrier()
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e4.record()
        for i in range(args.steps):
            step(dev_ids[args.warmup + i])
        e5.record()
        barrier()
        ms_nockpt = e4.elapsed_time(e5)
        model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    # ---- extra: the same step with one library GEMM per q/k/v module (A/B of the fused dense kernels in the real step) ----
    ms_unfused = None
    if n_fused_layers and not args.no_extra:
        M.unfuse_qkv_projections(model)
        for i in range(2):
            step(dev_ids[i])
        barrier()
        e6, e7 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e6.record()
        for i in range(args.steps):
            step(dev_ids[args.warmup + i])
        e7.record()
        barrier()
        ms_unfused = e6.elapsed_time(e7)
        M.fuse_qkv_projections(model)
    # ---- cross-rank reductions of the timings ------------------------------------------------------------------------
    breakdown = {"phases": ["forward", "backward (incl. grouped block-grad GEMM chunks)", "exchange wait", "adam + zero_grad"],
                 "mean_ms_this_rank": phase_mean, "host_flush_ms_per_step": host_flush_ms,
                 # activations (x, dy of every converted module) that the deferred grouped launch keeps alive until it runs
                 "operand_bytes_held_until_flush_max": ops.HOST_TIME["operand_bytes_held_max"]}
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e, ms_nockpt or 0.0, ms_unfused or 0.0], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e, ms_nockpt, ms_unfused = t.tolist()
        ms_nockpt = ms_nockpt or None
        ms_unfused = ms_unfused or None
        mine = torch.tensor(phase_mean + [sum(phase_mean)], device=device, dtype=torch.float64)
        allp = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allp, mine)
        allp = torch.stack(allp)                                      # [rank, phase]
        clk = torch.tensor([clocks["sm_mhz"] or 0.0, 1.0 if "sw_power_cap" in clocks["reasons"] else 0.0],
                           device=device, dtype=torch.float64)
        allc = [torch.empty_like(clk) for _ in range(world)]
        dist.all_gather(allc, clk)
        breakdown.update(per_rank_mean_ms=allp[:, :4].tolist(), min_over_ranks=allp.min(0).values.tolist(),
                         max_over_ranks=allp.max(0).values.tolist(),
                         step_skew_ms=(allp[:, 4].max() - allp[:, 4].min()).item(), exchange=exch_ms,
                         per_rank_sm_mhz_median=[c[0].item() for c in allc],
                         per_rank_sw_power_cap=[bool(c[1].item()) for c in allc])

    # ---- config 5 (BASELINE configs[4] shape: attention + MLP blocks), driver-visible sub-record --------------------
    config5 = None
    if not args.no_extra and args.mlp_ratio == 0.0 and args.layers == 32:
        try:
            if exchange is not None:
                exchange.close()
            M.set_grouped_backward(False)
            model = M.convert_matrix_sparsity_to_linear_layer(model)
            del opt
            torch.cuda.empty_cache()
            set_capture_requires_grad(True)
            k5 = H.block_budget(model, CONFIG5_RATIO, BLOCK)
            a5, m5, _ = capture_phase(True, 1)
            s5a, s5m = select(a5, m5, k5, k5)
            del a5, m5
            opt5 = convert(s5a, s5m)
            if not args.no_fuse_qkv:
                M.fuse_qkv_projections(model)
            M.set_grouped_backward(not args.no_group, chunk_blocks=args.chunk_blocks if overlap else 0)
            ex5 = dp.OverlappedGradExchange(opt5) if overlap else None

            def step5(ids):
                out = model(input_ids=ids, labels=ids, use_cache=False)
                out.loss.backward()
                if ex5 is not None:
                    ex5.finish()
                else:
                    for w in dp.allreduce_compact_grads(opt5, async_op=True):
                        w.wait()
                opt5.step()
                opt5.zero_grad()
                return out.loss

            for i in range(3):
                step5(dev_ids[i])
            ops.enable_timing("block_grad_gemm")
            n5 = max(4, min(args.steps, 8))
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n5):
                l5 = step5(dev_ids[args.warmup + i % args.steps])
            b.record()
            barrier()
            ms5 = a.elapsed_time(b)
            g5 = ops.collect_timing("block_grad_gemm")
            ops.enable_timing("block_grad_gemm", False)
            ident5 = dp.replicas_identical(opt5) if world > 1 else None
            if world > 1:
                t = torch.tensor([ms5], device=device, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms5 = t.item()
            g5_ms = sum(ms for ms, _ in g5)
            g5_flops = sum(2.0 * tag[1] * tag[1] * tag[2] * tag[0] for _ms, tag in g5)
            config5 = {"workload": f"LLaMA-3-8B shape (= DeepSeek-R1-Distill-Llama-8B), SMT {200 * CONFIG5_RATIO:.2f}%: "
                                   f"{sum(len(v) for v in s5a.values())} attention + {sum(len(v) for v in s5m.values())} MLP "
                                   f"blocks, gradient-based selection (what the reference's published command runs), "
                                   f"bf16, seq {S} x batch {B} per GPU",
                       "value": B * S * world * n5 / (ms5 / 1e3), "unit": "tokens/s", "steps": n5, "warmup": 3,
                       "ms_per_step": ms5 / n5, "modules_with_blocks": len(s5a) + len(s5m),
                       "block_grad_gemm_tflops": g5_flops / (g5_ms * 1e-3) / 1e12 if g5_ms > 0 else None,
                       "block_grad_gemm_launches_per_step": len(g5) / n5, "loss_last": l5.item(),
                       "params_identical_across_ranks": ident5}
            if ex5 is not None:
                ex5.close()
        except Exception as e:  # the headline must survive a failure of this extra record
            config5 = {"error": f"{type(e).__name__}: {e}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    tokens = B * S * world * args.steps
    value = tokens / (ms_total / 1e3)
    e2e_value = tokens / (ms_e2e / 1e3)
    # ---- roofline of the dominant SMT kernel: block-gradient GEMM ---------------------------------------------------
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0         # sustained: the kernel is timed inside a long step
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
    gemm_ms = sum(ms for ms, _ in gemm_t)
    gemm_flops = sum(2.0 * tag[1] * tag[1] * tag[2] * tag[0] for _ms, tag in gemm_t)
    n_gemm = len(gemm_t)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0

    def x_group(kind):                                            # modules that read the same input activation
        return "attn" if kind in ("q_proj", "k_proj", "v_proj") else ("mlp_in" if kind in ("gate_proj", "up_proj") else kind)
    x_strips = {(x_group(k[0]), k[1], c) for k, idx in sel.items() for _r, c in idx}
    dy_strips = {(k, r) for k, idx in sel.items() for r, _c in idx}
    gemm_min_bytes = 2.0 * T * BLOCK * (len(x_strips) + len(dy_strips)) + 2.0 * n_blocks * BLOCK * BLOCK
    traffic, traffic_note = None, None
    for name in ("r02_bench_gemm_traffic.json", "r01_bench_gemm_traffic.json"):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", name)))
            if args.layers == 32 and not args.no_group and n_mlp == 0 and args.attn_ratio == ATTN_RATIO \
                    and os.environ.get("SMT_GEMM_2SM") != "0":
                traffic = (tr["dram_bytes_read"] + tr["dram_bytes_write"]) * tr.get("launches_per_step", 1) * args.steps \
                    / max(n_gemm, 1)
                traffic_note = (f"dram read+write bytes per launch from one ncu --set full capture of this workload at 1 GPU "
                                f"(profiles/{name}; the per-rank work is identical at every N); algorithmic minimum in "
                                "min_hbm_bytes_per_launch")
            break
        except Exception:
            continue
    adam_ms = statistics.mean(ms for ms, _ in adam_t) if adam_t else None
    gemm_kernel = "block_grad_umma_kernel<256, 2, grouped> (single-CTA tiles)" if os.environ.get("SMT_GEMM_2SM") == "0" \
        else "block_grad_umma_2sm_kernel (cta_group::2, two 256x256 blocks per SM pair)"
    also = {"compact_adam": {"bound": "hbm", "avg_ms": adam_ms,
                             "achieved_gbs": (trainable * 30 / (adam_ms * 1e-3) / 1e9) if adam_ms else None,
                             "peak_gbs": hbm_peak, "bytes_per_elem": 30,
                             "frac": (trainable * 30 / (adam_ms * 1e-3) / 1e9 / hbm_peak) if adam_ms else None,
                             "clip_norm_source": sq_source}}
    if score_roof:
        also.update(score_roof if "error" not in score_roof else {"score_kernels": score_roof})
    if cfg2:
        also["config2"] = cfg2
    if qkv_ab:
        also["fused_qkv"] = qkv_ab
    roofline = {"kernel": gemm_kernel, "bound": "tensor", "achieved": achieved,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                "traffic_note": traffic_note,
                "min_hbm_bytes_per_launch": gemm_min_bytes * args.steps / max(n_gemm, 1),
                "frac_of_burst_peak": achieved / peaks.get("bf16_tflops", 1599.5),
                "peak_source": peak_src, "launches": n_gemm, "avg_launch_us": gemm_ms * 1e3 / max(n_gemm, 1),
                "flops_per_launch": gemm_flops / max(n_gemm, 1), "share_of_step": gemm_ms / ms_total,
                "also": also}
    smt_ms_per_step = (gemm_ms + sum(ms for ms, _ in adam_t)) / max(args.steps, 1)
    dense_ms = sum(ms for ms, _ in fwd_t) + sum(ms for ms, _ in dgr_t)
    dense_flops = sum(2.0 * t[0] * t[1] * t[2] for _ms, t in fwd_t) + sum(2.0 * t[0] * t[1] * t[2] for _ms, t in dgr_t)
    if dense_ms > 0:
        also.setdefault("fused_qkv", {})["in_step"] = {
            "launches_per_step": (len(fwd_t) + len(dgr_t)) / max(args.steps, 1),
            "ms_per_step": dense_ms / max(args.steps, 1),
            "tflops": dense_flops / (dense_ms * 1e-3) / 1e12,
            "frac_of_sustained_peak": dense_flops / (dense_ms * 1e-3) / 1e12 / peak_tf,
            "share_of_step": dense_ms / ms_total}
    line = {"metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "per_gpu_value": value / world,
            "config": {"workload": (f"LLaMA-3-8B SMT {100 * (args.attn_ratio + args.mlp_ratio):.2f}% "
                                    + ("q/k/v" if n_mlp == 0 else "q/k/v + MLP")
                                    + f" gradient-based selection, bf16, seq {S} x batch {B} per GPU")
                                   + ("" if args.layers == 32 else f" [DEBUG: {args.layers} layers only]"),
                       "selected_blocks": n_blocks, "block": BLOCK, "trainable_elements": trainable,
                       "modules_with_blocks": len(sel), "grouped_block_grad_launch": not args.no_group,
                       "grouped_launch_shape": grouped_shape,
                       "fused_qkv_layers": n_fused_layers,
                       "total_blocks_budget_base": total_blocks, "gradient_checkpointing": not args.no_ckpt,
                       "parallelism": f"dp{world}", "tokens_per_step_per_gpu": T,
                       "gradient_exchange": ("none (1 GPU)" if world == 1 else
                                             (f"overlapped: grouped GEMM flushed every >= {args.chunk_blocks} blocks at layer "
                                              "boundaries, each chunk all-reduced (+ its sum of squares) on a side stream during "
                                              "backward" if overlap else "one blocking all-reduce after backward")),
                       "l2": "inputs larger than L2 (16 GB of weights streamed per step); no explicit flush",
                       "loss_last": last,
                       "tokens_per_s_without_checkpointing": (tokens / (ms_nockpt / 1e3)) if ms_nockpt else None,
                       "ms_per_step_with_library_qkv_gemms": (ms_unfused / args.steps) if ms_unfused else None,
                       # SMT-layer-only view: the step is dominated by the HF model's dense GEMMs and elementwise kernels
                       # (out of scope); this is what the in-scope kernels alone cost per step
                       "smt_kernels_ms_per_step": smt_ms_per_step,
                       "smt_kernels_share_of_step": smt_ms_per_step / (ms_total / args.steps),
                       "smt_kernels_only_tokens_per_s_per_gpu": T / (smt_ms_per_step / 1e3) if smt_ms_per_step > 0 else None,
                       "warmup_mode": (f"capture-only, no optimizer step (declared deviation from fine_tune.py:168-190, which "
                                       f"runs real full-FT steps under ZeRO + offload): {len(capture_ms)} gradient-capture "
                                       "passes, grad-ready hooks -> on-device block-sum accumulators, gradients released at "
                                       "once; the reference's full-FT policy is measured in warmup_full_ft_policy"),
                       "warmup_full_ft_policy": full_ft,
                       # warm-up times below (and the full-FT record's) describe this attention backward
                       "warmup_attention_backward": ("math (deterministic, --dump-outputs)" if args.dump_outputs
                                                     else "default SDPA kernel"),
                       "warmup_path_ms": {"capture_pass_first_cold": capture_ms[0],
                                          "capture_pass_steady": statistics.median(capture_ms[1:]) if len(capture_ms) > 1 else None,
                                          "same_pass_without_capture_hooks": plain_ms,
                                          "score_kernel_launches_per_pass": capture_launches / max(len(capture_ms), 1),
                                          "scores_topk": t_select * 1e3}},
            "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": B * S * 8, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "step_breakdown": breakdown}
    if dp_check is not None:
        dp_check["params_identical"] = params_identical
        line["dp_check"] = dp_check
    if config5 is not None:
        line["config5"] = config5
    if world == 1 and not args.no_cpu_baseline:
        try:
            tps, ms, cores, sample, kind = cpu_reference_arm(steps=3, warmup=1, seq=args.cpu_seq)
            line["cpu_baseline"] = {"value": tps, "unit": "tokens/s", "cores": cores, "kind": kind, "sample": sample,
                                    "measured_ms_per_layer_step": ms}
        except Exception as e:  # keep the GPU result even if the CPU leg cannot run
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"failed: {type(e).__name__}: {e}"}
    if world == 1 and not args.no_extra and args.layers == 32:
        line["secondary_comparator"] = eager_reference_on_gpu(args, model, dev_ids, sel_attn, device)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def eager_reference_on_gpu(args, model, dev_ids, sel_attn, device):
    """The speed-up that means something: the reference's OWN modules (oracle/_ref: unmodified `LinearLayer_MatrixSparsity`
    / `linearZ`, smt.py:302-413) converted into the same LLaMA-3-8B with the same 869 blocks and run eagerly ON THE B200
    for full steps of the same workload (batch x seq, gradient checkpointing), with torch's fused AdamW + clip_grad_norm_
    standing in for DeepSpeed's FusedAdam.  `model` arrives holding plain nn.Linear modules again."""
    import torch
    try:
        from sparse_matrix_tuning_b200.smt import smt as M
        ref_smt, kind = _reference_modules()
        if ref_smt is None:
            return {"unavailable": "oracle/_ref not staged (run oracle/build_ref.py where /root/reference exists)"}
        model = M.convert_matrix_sparsity_to_linear_layer(model)
        for p in model.parameters():
            p.requires_grad = False
        torch.cuda.empty_cache()
        n_conv = 0
        for (kind_name, layer), idx in sel_attn.items():
            attn = model.model.layers[layer].self_attn
            lin = getattr(attn, kind_name)
            setattr(attn, kind_name, ref_smt.LinearLayer_MatrixSparsity(lin.weight, bias=None, index_list=list(idx)))
            n_conv += 1
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-4, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.0, fused=True)
        model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
        model.enable_input_require_grads()
        model.train()

        def step(ids):
            out = model(input_ids=ids, labels=ids, use_cache=False)
            out.loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
            opt.zero_grad(set_to_none=False)
            return out.loss

        step(dev_ids[0])
        n = 3
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            loss = step(dev_ids[args.warmup + i % max(args.steps, 1)])
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / n
        return {"what": "reference's own smt.py modules (oracle/_ref, unmodified) run eagerly on this B200: same model, "
                        f"same {sum(len(v) for v in sel_attn.values())} blocks in {n_conv} modules, same batch x seq, "
                        "gradient checkpointing, torch fused AdamW + clip_grad_norm_ in place of DeepSpeed FusedAdam",
                "value": args.batch * args.seq / (ms / 1e3), "unit": "tokens/s", "ms_per_step": ms, "steps": n, "warmup": 1,
                "loss_last": loss.item()}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
