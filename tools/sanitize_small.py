"""Tiny end-to-end pass over every kernel for compute-sanitizer (memcheck): small shapes, all code paths
(whole/half-block tiles, fused and separate split-K reduction, grouped launch, fp32 path, Adam with write-back,
top-k shared/global sort, gather/scatter, score kernels; run tiles, per-item overwrite + sums of squares, channel gradient,
fused dense GEMMs, Adam with partial norms)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sparse_matrix_tuning_b200 import ops

torch.manual_seed(0)
dev = "cuda"
for b, T, n, fin, fout in ((256, 320, 2, 512, 512), (256, 1100, 3, 512, 768), (128, 600, 3, 512, 256), (64, 200, 5, 256, 256),
                           (256, 256, 160, 2560, 4096)):
    x = torch.randn(T, fin, device=dev).bfloat16()
    dy = torch.randn(T, fout, device=dev).bfloat16()
    perm = torch.randperm((fout // b) * (fin // b))[:n]
    idx = [(int(p) // (fin // b), int(p) % (fin // b)) for p in perm]
    rc = ops.make_block_rc(idx, dev)
    for env in ("0", "1"):
        os.environ["SMT_GEMM_NO_FUSED_REDUCE"] = env
        out = ops.block_grad_gemm(x, dy, rc, b, out_dtype=torch.bfloat16)
        out32 = torch.zeros(len(idx) * b, b, device=dev)
        ops.block_grad_gemm(x, dy, rc, b, out=out32, accumulate=True)
    os.environ["SMT_GEMM_NO_FUSED_REDUCE"] = "0"
    batch = ops.BlockGradBatch()
    flat = torch.zeros(2 * len(idx) * b * b, device=dev, dtype=torch.bfloat16)
    batch.add(x, dy, idx, flat[: len(idx) * b * b].view(-1, b), b)
    batch.add(x, dy, idx, flat[len(idx) * b * b:].view(-1, b), b)
    batch.flush()
    ref = dy.float()[:, idx[0][0] * b:(idx[0][0] + 1) * b].t() @ x.float()[:, idx[0][1] * b:(idx[0][1] + 1) * b]
    assert (out32[:b] - ref).abs().max() <= 2e-5 * ref.abs().max()
xf = torch.randn(2, 50, 256, device=dev)
ops.block_grad_gemm(xf.reshape(-1, 256), xf.reshape(-1, 256), ops.make_block_rc([(1, 0), (0, 1)], dev), 128)
W = torch.randn(512, 512, device=dev).bfloat16()
tab = ops.make_block_table([(W, 0, 1), (W, 1, 0)], dev)
comp = torch.empty(512, 256, device=dev, dtype=torch.bfloat16)
ops.block_gather(tab, 2, 256, comp)
ops.block_scatter(tab, 2, 256, comp)
N = 2 * 256 * 256
st = [torch.zeros(N, device=dev) for _ in range(3)]
g = torch.randn(N, device=dev).bfloat16()
sq = ops.grad_sqnorm(g)
ops.compact_adam(*st, g, lr=1e-3, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.01, step=1, sqnorm=sq, max_norm=1.0,
                 compact_out=comp.view(-1), table=tab, n_blocks=2, block=256, w_dtype=torch.bfloat16)
acc = torch.zeros(512, 768, device=dev)
ops.score_accumulate(acc, torch.randn(512, 768, device=dev).bfloat16())
for s in ("mean_abs", "L2"):
    ops.block_score_reduce(acc, 256, s)
sums = torch.zeros(2, 3, device=dev)
ops.block_sum_accumulate(sums, acc.bfloat16(), 256)
ops.block_sum_finalize(sums, 256)
a2 = torch.zeros(40, 256, device=dev)
ops.act_score_accumulate(a2, torch.randn(3, 40, 256, device=dev).bfloat16())
ops.channel_score_reduce(a2, "L1")
sc = torch.rand(30000, device=dev)
ops.topk_blocks(sc, [0, 30000], [100])
ops.topk_blocks(sc, [0, 10000, 30000], [9000, 17])
# round-2 kernels: per-item overwrite + sums of squares, run tiles, channel gradient, fused dense GEMMs, Adam with partials
for b in (64, 128, 256):
    T, fin = 300, 1024
    x = torch.randn(T, fin, device=dev).bfloat16()
    dy = torch.randn(T, fin, device=dev).bfloat16()
    nb = fin // b
    idx = [(r, c) for r in range(min(nb, 3)) for c in range(nb)]
    if b != 256:                                                    # run tiles exist for b = 64 / 128
        got = ops._gemm_runs(x, dy, ops._runs_for(idx, b, x.device), b,
                             torch.empty(len(idx) * b, b, device=dev), False)
        ref = dy.float()[:, :b].t() @ x.float()[:, :b]
        assert (got[:b] - ref).abs().max() <= 3e-5 * ref.abs().max()
    flat = torch.zeros(len(idx) * b * b, device=dev, dtype=torch.bfloat16)
    sqp = torch.zeros(2 * len(idx), device=dev)
    batch = ops.BlockGradBatch()
    batch.add(x, dy, idx, flat.view(-1, b), b, accumulate=False, sq=sqp, sq_slot0=0)
    batch.flush(accumulate=True)
xq = torch.randn(300, 512, device=dev).bfloat16()
ws = [torch.randn(n, 512, device=dev).bfloat16() for n in (512, 256, 256)]
ys = ops.fused_linear_forward(xq, ws)
dx = ops.fused_linear_dgrad([torch.randn_like(y) for y in ys], ws)
cidx = ops.make_channel_idx([3, 70, 500], dev, pad_to=8)
part = ops.channel_gather(xq, cidx)
ops.channel_grad_gemm(part, 3, torch.randn(300, 256, device=dev).bfloat16())
ops.compact_adam(*st, g, lr=1e-3, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.0, step=2,
                 sqnorm=torch.rand(300, device=dev), max_norm=1.0)
torch.cuda.synchronize()
print("sanitize_small: ok")
