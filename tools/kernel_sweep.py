"""BASELINE config 2: single-layer sweep of the block-gradient GEMM (per-module launch, `smt_block_grad_gemm`).

    weights {4096x4096 (q), 14336x4096 (gate/up), 4096x14336 (down)} x block {64,128,256} x sparsity {0.5,1,2,5} %
    x tokens {2048, 8192, 16384} (seq 2048 x batch 1/4/8), bf16, x,dy ~ N(0,1), blocks by seeded randperm,
    plus a "clustered" set (all blocks in one block-row) that exposes strip reuse.

Prints a markdown table: time (CUDA events, L2 flushed between iterations, median of 7), TFLOP/s, and the fraction
of the applicable roofline = max(flops / bf16 peak, min HBM bytes / HBM peak) (DESIGN.md section 3.1).
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sparse_matrix_tuning_b200 import ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
try:
    PEAKS = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
except Exception:
    PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")


def timeit(fn, iters=7, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2] * 1e-3     # seconds


def main():
    quick = "--quick" in sys.argv
    shapes = [(4096, 4096, "q 4096x4096"), (14336, 4096, "gate/up 14336x4096"), (4096, 14336, "down 4096x14336")]
    tokens = [2048, 8192, 16384] if not quick else [8192]
    print("| weight [out x in] | b | sparsity | pattern | T | n | kernel | us | us (block tiles only) | us (run tiles forced) | TFLOP/s | of bf16 burst peak | roofline bound | of roofline |")
    print("|---|---:|---:|---|---:|---:|---|---:|---:|---:|---:|---:|---|---:|")
    g = torch.Generator().manual_seed(1234)
    for fout, fin, label in shapes:
        for T in tokens:
            x = torch.randn(T, fin, device="cuda").bfloat16()
            dy = torch.randn(T, fout, device="cuda").bfloat16()
            for b in (256, 128, 64):
                total = (fout // b) * (fin // b)
                for sp in (0.005, 0.01, 0.02, 0.05):
                    n = max(1, int(sp * total))
                    for pattern in ("random", "clustered"):
                        if pattern == "random":
                            perm = torch.randperm(total, generator=g)[:n]
                            idx = [(int(p) // (fin // b), int(p) % (fin // b)) for p in perm]
                        else:
                            if n > fin // b or sp not in (0.01, 0.05):
                                continue
                            idx = [(1, c) for c in range(n)]
                        rc = ops.make_block_rc(idx, "cuda")
                        out = torch.empty(n * b, b, device="cuda", dtype=torch.bfloat16)
                        # round-1 kernel: one tile per block; run tiles forced (b = 64 / 128 only)
                        t_blocks = timeit(lambda: ops._gemm_blocks(x, dy, rc, b, out, False))
                        runs_us = "-"
                        if b != 256:
                            t_runs = timeit(lambda: ops._gemm_runs(x, dy, ops._runs_for(idx, b, x.device), b, out, False))
                            runs_us = f"{t_runs * 1e6:.1f}"
                        # default: strip-sharing runs when they pay
                        t = timeit(lambda: ops.block_grad_gemm(x, dy, rc, b, out=out, index_list=idx))
                        kern = ops.LAST_SINGLE.get("kernel", "?")
                        flops = 2.0 * b * b * T * n
                        ur, uc = len({r for r, _ in idx}), len({c for _, c in idx})
                        min_bytes = 2.0 * T * b * (ur + uc) + n * b * b * 2
                        t_tensor = flops / (PEAKS["bf16_tflops"] * 1e12)
                        t_hbm = min_bytes / (PEAKS["hbm_gbs"] * 1e9)
                        bound = "tensor" if t_tensor >= t_hbm else "hbm"
                        print(f"| {label} | {b} | {sp * 100:g}% | {pattern} | {T} | {n} | {kern} | {t * 1e6:.1f} | {t_blocks * 1e6:.1f} | {runs_us} | "
                              f"{flops / t / 1e12:.1f} | {flops / t / 1e12 / PEAKS['bf16_tflops']:.3f} | {bound} | "
                              f"{max(t_tensor, t_hbm) / t:.3f} |", flush=True)
            del x, dy


if __name__ == "__main__":
    main()
