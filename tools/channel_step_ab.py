"""A/B of the channel-sparse training step on one GPU, in one process; prints one JSON object (and writes it to --out).

Workload: LLaMA-3-8B in bf16, B 16 x S 512, recomputation on (non-reentrant checkpointing), `--channels` (default 288)
random input channels in every q/k/v module: 96 LinearLayer_ChannelSparsity modules, 56.6 M trainable elements at 288.

  native  SMTAdam arena with channel owners (gradients delivered into the arena by grouped launches, one
          smt_compact_adam_columns launch with the column write-back), fuse_qkv_projections (fused dense q/k/v GEMMs and
          the decoder-layer kernels);
  today   the per-module path: a channel_grad_gemm per module into a fresh tensor copied into the arena, a grad_sqnorm
          pass, one compact_adam per parameter, a column_scatter in every forward, HF elementwise ops.

The two arms run on two identical models, alternating A B A B; per arm: ms/step (CUDA events around `--steps` steps),
SMT kernel launches per step, max_memory_allocated above the memory held when the arm starts.  During the native arm the
Adam-columns kernel is bracketed by CUDA events (the forward and backward of the step evict the L2 between two launches)
and its time is set against two lower bounds at `--hbm-gbs`: 30 B/element of state traffic (bf16 grad 2, fp32 master,
exp_avg, exp_avg_sq 3 x 8, bf16 compact copy 2, bf16 weight 2) and 60 B/element when every weight store costs a whole
32-byte sector (the 2-byte column stores are one weight row apart).

    python tools/channel_step_ab.py --out /tmp/r06_channel_native_step_raw.json
    python tools/channel_step_ab.py --dry-run          # element and byte counts only, no GPU
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

HID, INTER, NQ, NKV, HD, LAYERS = 4096, 14336, 32, 8, 128, 32
LLAMA3_8B = dict(vocab_size=128256, hidden_size=HID, intermediate_size=INTER, num_hidden_layers=LAYERS,
                 num_attention_heads=NQ, num_key_value_heads=NKV, max_position_embeddings=8192, rms_norm_eps=1e-5,
                 rope_theta=500000.0, attn_implementation="sdpa")
OUT_FEATURES = {"q_proj": NQ * HD, "k_proj": NKV * HD, "v_proj": NKV * HD}


def counts(channels: int) -> dict:
    elems = LAYERS * channels * sum(OUT_FEATURES.values())
    return {"modules": 3 * LAYERS, "trainable_elements": elems, "state_bytes": 30 * elems,
            "sector_bound_bytes": 60 * elems}


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [s.strip() for s in out[0].split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as e:  # reported, not fatal: the timings still carry the device name from torch
        return {"error": f"{type(e).__name__}: {e}"}


# SMT entry points whose calls are counted per step, by name (each is one kernel launch, grad_sqnorm two; a grouped or
# channel gradient launch may add a split-K reduction, which the total of ops.LAUNCHES includes)
COUNTED = ("channel_gather", "column_scatter", "channel_grad_gemm", "grad_sqnorm", "compact_adam", "fused_linear_forward",
           "fused_linear_dgrad", "rmsnorm_forward", "rmsnorm_backward", "rope_forward", "rope_backward",
           "swiglu_forward", "swiglu_backward")


def count_calls(calls: dict) -> None:
    from sparse_matrix_tuning_b200 import ops

    def wrap(name, fn):
        def counted(*a, **k):
            calls[name] = calls.get(name, 0) + 1
            return fn(*a, **k)
        return counted

    for name in COUNTED:
        setattr(ops, name, wrap(name, getattr(ops, name)))
    ops.BlockGradBatch._launch_group = wrap("grouped_gradient_launch", ops.BlockGradBatch._launch_group)


def build_arm(native: bool, channels: int):
    import random

    import torch
    from transformers import LlamaConfig, LlamaForCausalLM
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
    sel = {(kind, l): sorted(rng.sample(range(HID), channels)) for l in range(LAYERS) for kind in OUT_FEATURES}
    M.freeze_unselected_channel_layer(model, {}, sel)
    M.convert_linear_layer_to_channel_sparsity(model, {}, sel)
    model.gradient_checkpointing_enable(gradient_checkpointing_kwargs={"use_reentrant": False})
    model.enable_input_require_grads()
    model.train()
    if not native:                                  # no owner: the arena treats the channels as plain parameters
        for m in model.modules():
            if isinstance(m, M.LinearLayer_ChannelSparsity):
                m._arena_ok = lambda: False
    opt = SMTAdam(M.get_optimizer_sparse_grouped_parameters(model, 0.0, 1e-4), lr=1e-4, betas=(0.9, 0.95),
                  max_grad_norm=1.0)
    if native:
        assert opt._arenas[0].all_sinks and opt._arenas[0].fused_writeback() is not None
    return model, opt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=288)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--seq", type=int, default=512)
    ap.add_argument("--steps", type=int, default=6, help="timed steps per arm and repetition")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--hbm-gbs", type=float, default=7700.0, help="HBM bandwidth the bounds refer to (data sheet)")
    ap.add_argument("--out", default="")
    ap.add_argument("--dry-run", action="store_true", help="print the element and byte counts, touch no GPU")
    args = ap.parse_args()
    if args.dry_run:
        print(json.dumps({"channels": args.channels, **counts(args.channels)}))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200.smt import smt as M
    t0 = time.time()
    result = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "channels": args.channels,
              "batch": args.batch, "seq": args.seq, **counts(args.channels), "hbm_gbs_reference": args.hbm_gbs}
    calls: dict = {}
    count_calls(calls)
    arms = {"native": build_arm(True, args.channels), "today": build_arm(False, args.channels)}
    gen = torch.Generator().manual_seed(0)
    ids = [torch.randint(0, LLAMA3_8B["vocab_size"], (args.batch, args.seq), generator=gen).cuda()
           for _ in range(args.steps)]

    def step(model, opt, t):
        loss = model(input_ids=t, labels=t, use_cache=False).loss
        loss.backward()
        opt.step()
        opt.zero_grad()
        return loss

    res = {arm: {"ms_per_step": [], "launches_per_step": [], "peak_bytes_above_start": [], "first_loss": None,
                 "calls_per_step": {}} for arm in arms}
    adam_ms = []
    for _ in range(args.reps):
        for arm, (model, opt) in arms.items():
            native = arm == "native"
            if native:
                assert M.fuse_qkv_projections(model) == LAYERS
            M.set_grouped_backward(native)
            for i in range(2):
                loss = step(model, opt, ids[i])
                if res[arm]["first_loss"] is None:
                    res[arm]["first_loss"] = loss.item()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            start = torch.cuda.memory_allocated()
            n0 = ops.LAUNCHES["total"]
            calls.clear()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for t in ids:
                step(model, opt, t)
            b.record()
            torch.cuda.synchronize()
            res[arm]["ms_per_step"].append(a.elapsed_time(b) / len(ids))
            res[arm]["launches_per_step"].append((ops.LAUNCHES["total"] - n0) / len(ids))
            res[arm]["calls_per_step"] = {k: v / len(ids) for k, v in sorted(calls.items())}
            res[arm]["peak_bytes_above_start"].append(torch.cuda.max_memory_allocated() - start)
            if native:                               # the Adam-columns kernel, in steps of its own (events on)
                ops.enable_timing("compact_adam_columns")
                for t in ids[:3]:
                    step(model, opt, t)
                torch.cuda.synchronize()
                adam_ms += [ms for ms, _tag in ops.collect_timing("compact_adam_columns")]
                ops.enable_timing("compact_adam_columns", False)
                M.unfuse_qkv_projections(model)
            M.set_grouped_backward(False)
    for arm in res:
        res[arm]["ms_per_step_median"] = statistics.median(res[arm]["ms_per_step"])
        res[arm]["max_memory_allocated_gb"] = max(res[arm]["peak_bytes_above_start"]) / 1e9
    result["arms"] = res
    result["speedup_min_over_pairs"] = min(t / n for t, n in zip(res["today"]["ms_per_step"],
                                                                 res["native"]["ms_per_step"]))
    t_adam = statistics.median(adam_ms) * 1e-3
    c = counts(args.channels)
    result["adam_columns"] = {
        "launch_ms": [round(x, 4) for x in adam_ms], "ms_median": t_adam * 1e3,
        "state_gb_per_s": c["state_bytes"] / t_adam / 1e9,
        "fraction_of_state_bound": c["state_bytes"] / (args.hbm_gbs * 1e9) / t_adam,
        "fraction_of_sector_bound": c["sector_bound_bytes"] / (args.hbm_gbs * 1e9) / t_adam}
    result["wall_s"] = time.time() - t0
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
