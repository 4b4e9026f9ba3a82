"""GPU parity tests, kernel level: every C-ABI entry point against the CPU oracle on the same seeded inputs.
Bars: bit-exact for integer / index / byte work (top-k indices, gather, scatter, Adam fp32 state vs the numpy
restatement); stated tolerances for floating-point reductions and the GEMM."""
import numpy as np
import pytest
import torch

from oracle import smt_oracle as O

pytestmark = pytest.mark.gpu

STRATEGIES = ("mean_abs", "abs_mean", "L1", "L2")


@pytest.fixture(scope="module")
def ops(built_library):
    from sparse_matrix_tuning_b200 import ops as _ops
    return _ops


# ---- scoring ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("block", [64, 128, 256])
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_block_score_reduce_vs_oracle(ops, block, strategy):
    torch.manual_seed(block)
    g = torch.randn(1024, 768)
    ref = O.block_scores(g, block, strategy)
    out = ops.block_score_reduce(g.cuda(), block, strategy).cpu()
    if strategy == "mean_abs":
        # signed sum: cancellation makes a relative bound meaningless; bound against the block's mean |g| instead
        scale = O.block_scores(g, block, "abs_mean")
        assert ((out - ref).abs() <= 2e-6 * scale).all()
    else:
        assert torch.allclose(out, ref, rtol=2e-6, atol=0)      # fp32 reduction-order tolerance


def test_block_score_reduce_strided_and_exact_cases(ops):
    base = torch.zeros(512, 1024, device="cuda")
    view = base[:, 256:768]                                      # ld = 1024, 512 columns
    view[:256, :256] = 3.0
    view[256:, 256:] = -2.0
    for s, want in (("mean_abs", [[3.0, 0.0], [0.0, 2.0]]), ("L1", [[3.0 * 65536, 0.0], [0.0, 2.0 * 65536]]),
                    ("L2", [[3.0 * 256, 0.0], [0.0, 2.0 * 256]])):
        assert ops.block_score_reduce(view, 256, s).cpu().tolist() == want


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_score_accumulate_matches_capture_loop(ops, dtype):
    """fine_tune.py:729-765: acc = sum over steps of grad.float()  (exact: same fp32 adds in the same order)."""
    torch.manual_seed(1)
    acc = torch.zeros(256, 520, device="cuda")
    ref = torch.zeros(256, 520)
    for _ in range(3):
        g = torch.randn(256, 520).to(dtype)
        ops.score_accumulate(acc, g.cuda())
        ref += g.float()
    assert torch.equal(acc.cpu(), ref)
    odd = torch.zeros(1003, device="cuda")
    g = torch.randn(1003).to(dtype)
    ops.score_accumulate(odd, g.cuda())
    assert torch.equal(odd.cpu(), g.float())


@pytest.mark.parametrize("block", [64, 256, 128])
def test_block_sum_mode_reproduces_mean_abs(ops, block):
    torch.manual_seed(2)
    sums = torch.zeros(512 // block, 768 // block, device="cuda")
    total = torch.zeros(512, 768)
    for _ in range(4):
        g = torch.randn(512, 768).bfloat16()
        ops.block_sum_accumulate(sums, g.cuda(), block)
        total += g.float()
    ref = O.block_scores(total, block, "mean_abs")
    scale = O.block_scores(total, block, "abs_mean")
    got = ops.block_sum_finalize(sums, block).cpu()
    assert ((got - ref).abs() <= 1e-5 * scale).all()


def test_activation_scoring_vs_oracle(ops):
    torch.manual_seed(3)
    steps = [torch.randn(3, 40, 512).bfloat16() for _ in range(2)]
    acc = torch.zeros(40, 512, device="cuda")
    for x in steps:
        ops.act_score_accumulate(acc, x.cuda())
    full = sum(x.float().abs() for x in steps)                   # what the reference hook accumulates, [B, S, C]
    assert torch.allclose(acc.cpu(), full.sum(0), rtol=1e-6, atol=1e-6)
    for s in STRATEGIES:
        ref = O.channel_scores(full, s)
        assert torch.allclose(ops.channel_score_reduce(acc, s).cpu(), ref, rtol=1e-5, atol=1e-6)


# ---- top-k: exact --------------------------------------------------------------------------------------

def _oracle_topk(scores_by_key, n):
    return O.select_from_scores(scores_by_key, n, "no_restriction")


@pytest.mark.parametrize("n_sel", [1, 7, 869, 5000])
def test_topk_indices_exact_with_ties(ops, n_sel):
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    torch.manual_seed(n_sel)
    keys = [(m, l) for l in (0, 1, 2, 10, 11) for m in ("q_proj", "k_proj", "v_proj")]
    scores = {}
    for m, l in keys:
        shape = (16, 16) if m == "q_proj" else (4, 16)
        s = torch.randn(shape).abs()
        s[torch.rand(shape) < 0.4] = 0.5                          # many exact ties across and inside matrices
        scores[(m, l)] = s
    n_sel = min(n_sel, sum(s.numel() for s in scores.values()))
    ref = _oracle_topk(scores, n_sel)
    got = H.select_submatrix_from_scores(list(scores), [s.cuda() for s in scores.values()], n_sel)
    assert list(got.items()) == list(ref.items())                 # same keys, same order, same (row, col) order


def test_topk_llama8b_size(ops):
    """12 288 q/k/v block scores, n = 869 (LLaMA-3-8B at 0.71 %) and 98 304 with MLP, n = 2106."""
    for total, n in ((12288, 869), (98304, 2106)):
        g = torch.Generator().manual_seed(total)
        sc = torch.rand(total, generator=g)
        sc[::5] = 0.25
        rank = torch.randperm(total, generator=g).int()
        inv = torch.empty_like(rank)
        inv[rank.long()] = torch.arange(total, dtype=torch.int32)
        idx, _ = ops.topk_blocks(sc.cuda(), [0, total], [n], rank.cuda(), inv.cuda())
        order = sorted(range(total), key=lambda i: (sc[i].item(), rank[i].item()), reverse=True)[:n]
        assert idx.cpu().tolist() == order


def test_topk_segments_and_degenerate_sizes(ops):
    g = torch.Generator().manual_seed(9)
    sc = torch.randn(3000, generator=g)
    offs, ks = [0, 1000, 1000, 2500, 3000], [10, 5, 2000, 7]
    idx, oo = ops.topk_blocks(sc.cuda(), offs, ks)
    vals = sc.tolist()
    for s in range(4):
        want = [i for _, i in sorted(((vals[i], i) for i in range(offs[s], offs[s + 1])), reverse=True)[:ks[s]]]
        assert idx[oo[s]:oo[s + 1]].cpu().tolist() == want
    assert oo == [0, 10, 10, 1510, 1517]
    big = torch.randn(40000, generator=g)                          # winners exceed shared memory: global-memory sort
    idx, _ = ops.topk_blocks(big.cuda(), [0, 40000], [20000])
    want = [i for _, i in sorted(((v, i) for i, v in enumerate(big.tolist())), reverse=True)[:20000]]
    assert idx.cpu().tolist() == want
    neg0 = torch.tensor([0.0, -0.0, 0.0, -0.0])                    # -0.0 == +0.0 in the reference's comparison
    idx, _ = ops.topk_blocks(neg0.cuda(), [0, 4], [4])
    assert idx.cpu().tolist() == [3, 2, 1, 0]


# ---- gather / scatter: byte-exact -------------------------------------------------------------------------

@pytest.mark.parametrize("block", [64, 128, 256])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32, torch.float16])
def test_gather_scatter_vs_oracle(ops, block, dtype):
    torch.manual_seed(block)
    w = torch.randn(512, 768).to(dtype)
    idx = [(1, 2), (0, 0), (512 // block - 1, 768 // block - 2), (0, 1)]     # distinct targets for every block size
    wd = w.cuda()
    tab = ops.make_block_table([(wd, r, c) for r, c in idx], "cuda")
    comp = torch.empty(len(idx) * block, block, dtype=dtype, device="cuda")
    ops.block_gather(tab, len(idx), block, comp)
    assert torch.equal(comp.cpu(), O.gather_blocks(w, idx, block))
    new = torch.randn_like(comp)
    ops.block_scatter(tab, len(idx), block, new)
    assert torch.equal(wd.cpu(), O.scatter_blocks(w.clone(), new.cpu(), idx, block))
    ops.block_gather(tab, len(idx), block, comp)                   # round trip
    assert torch.equal(comp, new)


# ---- optimizer ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("grad_dtype", [torch.bfloat16, torch.float32, torch.float16])
def test_compact_adam_bit_exact_vs_numpy_restatement(ops, grad_dtype):
    """fp32 master / exp_avg / exp_avg_sq after each step are BIT-IDENTICAL to oracle.adamw_fused_step (every op
    individually rounded), including the in-kernel clip coefficient; bf16 outputs are the RNE rounding of the master."""
    rng = np.random.RandomState(7)
    block, n_blocks = 64, 6
    N = n_blocks * block * block
    W = torch.randn(256, 256).bfloat16().cuda()
    idx = [(i // 4, i % 4) for i in range(n_blocks)]
    tab = ops.make_block_table([(W, r, c) for r, c in idx], "cuda")
    p = (rng.randn(N) * 0.02).astype(np.float32)
    m = np.zeros(N, np.float32)
    v = np.zeros(N, np.float32)
    dp, dm, dv = (torch.from_numpy(a.copy()).cuda() for a in (p, m, v))
    comp = torch.empty(N, dtype=torch.bfloat16, device="cuda")
    hp = dict(lr=3e-4, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.01)
    for step in range(1, 5):
        g = torch.from_numpy((rng.randn(N) * (0.05 if step % 2 else 1e-4)).astype(np.float32)).to(grad_dtype)
        gd = g.cuda()
        sq = ops.grad_sqnorm(gd)
        gscale = O.clip_coef(np.float32(sq.item()), np.float32(0.5), np.float32(1.0))
        ops.compact_adam(dp, dm, dv, gd, step=step, grad_scale=0.5, sqnorm=sq, max_norm=1.0, compact_out=comp,
                         table=tab, n_blocks=n_blocks, block=block, w_dtype=torch.bfloat16, **hp)
        p, m, v = O.adamw_fused_step(p, m, v, g.float().numpy(), step=step, gscale=gscale, **hp)
        assert np.array_equal(dp.cpu().numpy(), p), f"master differs at step {step}"
        assert np.array_equal(dm.cpu().numpy(), m) and np.array_equal(dv.cpu().numpy(), v)
        assert np.array_equal(comp.float().cpu().numpy(), O.bf16_round(p))
        assert torch.equal(O.gather_blocks(W.cpu(), idx, block).reshape(-1), comp.cpu())   # fused write-back
    # sum of squares vs float64
    ref_sq = float((g.double() ** 2).sum())
    assert abs(sq.item() - ref_sq) <= 1e-5 * ref_sq


def test_grad_sqnorm_is_deterministic(ops):
    g = torch.randn(3_000_001, device="cuda").bfloat16()
    a = ops.grad_sqnorm(g).item()
    for _ in range(3):
        assert ops.grad_sqnorm(g).item() == a
    assert abs(a - float((g.double() ** 2).sum())) <= 1e-5 * a


# ---- block-gradient GEMM --------------------------------------------------------------------------------------

def _gemm_inputs(B, S, fin, fout, block, n, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, S, fin, generator=g).to(dtype)
    dy = torch.randn(B, S, fout, generator=g).to(dtype)
    perm = torch.randperm((fout // block) * (fin // block), generator=g)[:n]
    idx = [(int(p) // (fin // block), int(p) % (fin // block)) for p in perm]
    return x, dy, idx


@pytest.mark.parametrize("block", [64, 128, 256])
@pytest.mark.parametrize("B,S", [(1, 64), (2, 100), (4, 512)])
def test_block_grad_gemm_bf16_vs_oracle(ops, block, B, S):
    """Tolerance (SURVEY §8c): bf16 result within 2^-7 of the tensor max of the fp64 truth AND no worse than the
    reference's own bf16 arithmetic (per-batch bmm rounded to bf16, then summed in bf16)."""
    x, dy, idx = _gemm_inputs(B, S, 1024, 768, block, 5, torch.bfloat16, seed=block + S)
    truth = O.block_grad_truth(x, dy, idx, block)
    _gi, ref = O.linearz_backward(x, dy, torch.zeros(768, 1024, dtype=torch.bfloat16), idx, block)
    out = ops.block_grad_gemm(x.cuda().reshape(-1, 1024), dy.cuda().reshape(-1, 768),
                              ops.make_block_rc(idx, "cuda"), block, out_dtype=torch.bfloat16).cpu()
    scale = truth.abs().max().item()
    err = (out.double() - truth).abs().max().item() / scale
    ref_err = (ref.double() - truth).abs().max().item() / scale
    assert err <= 2 ** -7
    # max statistic: 10 % slack (for B == 1 both are one rounding of nearly the same fp32 sum); mean: none
    assert err <= ref_err * 1.10 + 1e-6, (err, ref_err)
    assert (out.double() - truth).abs().mean() <= (ref.double() - truth).abs().mean() * 1.001
    # fp32 output of the same launch: only the fp32 accumulation error remains
    out32 = ops.block_grad_gemm(x.cuda().reshape(-1, 1024), dy.cuda().reshape(-1, 768),
                                ops.make_block_rc(idx, "cuda"), block, out_dtype=torch.float32).cpu()
    assert (out32.double() - truth).abs().max().item() / scale <= 1e-5


@pytest.mark.parametrize("block", [64, 128, 256])
def test_block_grad_gemm_fp32_vs_oracle(ops, block):
    """fp32 models (BASELINE config 1): 1e-5 of the tensor max, the tolerance north_star's fp32 parity implies."""
    x, dy, idx = _gemm_inputs(2, 77, 512, 512, block, 4, torch.float32, seed=block)
    _gi, ref = O.linearz_backward(x, dy, torch.zeros(512, 512), idx, block)
    out = ops.block_grad_gemm(x.cuda().reshape(-1, 512), dy.cuda().reshape(-1, 512),
                              ops.make_block_rc(idx, "cuda"), block).cpu()
    assert (out - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()


@pytest.mark.parametrize("block", [64, 256])
def test_block_grad_gemm_split_k_accumulate_and_strides(ops, block):
    x, dy, idx = _gemm_inputs(1, 4096 + 40, 1024, 512, block, 3, torch.bfloat16, seed=5)
    truth = O.block_grad_truth(x, dy, idx, block)
    scale = truth.abs().max().item()
    xd, dyd = x.cuda().reshape(-1, 1024), dy.cuda().reshape(-1, 512)
    rc = ops.make_block_rc(idx, "cuda")
    splits, _ = ops.block_grad_gemm_plan(len(idx), block, xd.shape[0], torch.bfloat16)
    assert splits > 1                                              # this case exercises the workspace + reduce path
    base = torch.randn(len(idx) * block, block, device="cuda")
    out = base.clone()
    ops.block_grad_gemm(xd, dyd, rc, block, out=out, accumulate=True)
    assert ((out.cpu().double() - base.cpu().double()) - truth).abs().max().item() / scale <= 2e-5
    # column-sliced (strided) operands: ld > features
    xs, dys = xd[:, 256:768], dyd[:, 128:384] if block == 64 else dyd[:, 0:256]
    idx2 = [(0, 1), ((256 // block) - 1, (512 // block) - 1)]
    got = ops.block_grad_gemm(xs, dys, ops.make_block_rc(idx2, "cuda"), block, out_dtype=torch.float32).cpu()
    t2 = O.block_grad_truth(xs.cpu(), dys.cpu(), idx2, block)
    assert (got.double() - t2).abs().max().item() / t2.abs().max().item() <= 2e-5
    # run-to-run determinism of the split-K path (fixed-order reduction, no atomics)
    a = ops.block_grad_gemm(xd, dyd, rc, block, out_dtype=torch.float32)
    b = ops.block_grad_gemm(xd, dyd, rc, block, out_dtype=torch.float32)
    assert torch.equal(a, b)


def test_block_grad_gemm_empty_inputs(ops):
    rc = ops.make_block_rc([(0, 0)], "cuda")
    x = torch.empty(0, 256, device="cuda", dtype=torch.bfloat16)
    out = ops.block_grad_gemm(x, x, rc, 256, out_dtype=torch.float32)
    assert out.shape == (256, 256) and not out.any()               # T == 0: the sum over no tokens is zero
    none = ops.block_grad_gemm(torch.zeros(8, 256, device="cuda", dtype=torch.bfloat16),
                               torch.zeros(8, 256, device="cuda", dtype=torch.bfloat16),
                               ops.make_block_rc([], "cuda"), 256)
    assert none.numel() == 0                                       # no selected block: nothing to do


def test_warmup_accumulator_vs_capture_loop(ops):
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    from sparse_matrix_tuning_b200.warmup import WarmupGradAccumulator
    torch.manual_seed(11)
    names = [f"model.layers.{l}.self_attn.{m}.weight" for l in (0, 1) for m in ("q_proj", "k_proj", "v_proj", "o_proj")]
    names += ["model.layers.0.mlp.up_proj.weight", "model.embed_tokens.weight"]
    shapes = {"q_proj": (512, 512), "k_proj": (256, 512), "v_proj": (256, 512), "o_proj": (512, 512),
              "up_proj": (768, 512), "embed_tokens": (1024, 512)}
    acc_e = WarmupGradAccumulator(block=256, mode="elementwise")
    acc_b = WarmupGradAccumulator(block=256, mode="block_sum")
    ref = {}
    for _step in range(3):
        grads = {n: torch.randn(*shapes[[k for k in shapes if k in n][0]]).bfloat16() for n in names}

        class P:  # minimal stand-in for a parameter with .grad
            def __init__(self, g):
                self.grad = g
        params = [(n, P(g.cuda())) for n, g in grads.items()]
        acc_e.accumulate(params)
        acc_b.accumulate(params)
        O.warmup_accumulate(ref, grads.items(), mlp=False, attention=True)
    assert list(acc_e.grads().keys()) == list(ref.keys())          # o_proj, MLP and embeddings are not captured
    for k in ref:
        assert torch.equal(acc_e.grads()[k].cpu(), ref[k])
    dims = {"q_proj": [512, 512], "k_proj": [256, 512], "v_proj": [256, 512]}
    want = O.select_submatrix(ref, dims, 6)
    assert list(H.select_submatrix_based_on_grads(acc_e.grads(), dims, 6).items()) == list(want.items())
    keys, scores = acc_b.scores("mean_abs")
    assert list(H.select_submatrix_from_scores(keys, scores, 6).items()) == list(want.items())


@pytest.mark.parametrize("block", [64, 256])
def test_grouped_gemm_matches_per_problem_launches(ops, block):
    """Several (x, dy) problems — q/k/v of one layer share x — in ONE grouped launch, accumulated into views of one
    flat buffer, against the per-problem launches and the fp64 truth."""
    torch.manual_seed(block)
    T, fin = 1000, 1024
    x = torch.randn(T, fin).bfloat16()
    dys = [torch.randn(T, fo).bfloat16() for fo in (1024, 512, 512)]
    x2 = torch.randn(T, fin).bfloat16()                              # a second "layer"
    dy2 = torch.randn(T, 1024).bfloat16()
    problems = [(x, dys[0], [(0, 1), (2, 3), (1, 1)]), (x, dys[1], [(1, 0)]), (x, dys[2], [(0, 2), (1, 3)]),
                (x2, dy2, [(3, 0), (0, 0), (2, 2), (1, 2)])]
    if block == 64:
        problems = [(a, d, [(r * 2 + 1, c * 3) for r, c in idx]) for a, d, idx in problems]
    total = sum(len(p[2]) for p in problems)
    flat = torch.randn(total * block * block, device="cuda")         # pre-existing content: accumulate on top
    base = flat.clone()
    batch = ops.BlockGradBatch()
    xd = {id(x): x.cuda(), id(x2): x2.cuda()}
    off, views, truths = 0, [], []
    for a, d, idx in problems:
        n = len(idx) * block * block
        view = flat[off:off + n].view(len(idx) * block, block)
        batch.add(xd[id(a)], d.cuda(), idx, view, block)
        views.append((off, n))
        truths.append(O.block_grad_truth(a, d, idx, block))
        off += n
    assert batch.flush(accumulate=True) == 1 and len(batch) == 0
    got = (flat - base).cpu().double()
    truth = torch.cat([t.reshape(-1) for t in truths])
    scale = truth.abs().max().item()
    assert (got - truth).abs().max().item() <= 3e-5 * scale          # fp32 accumulate, fp32 output (+ the fp32 add)
    for (a, d, idx), (o, n) in zip(problems, views):
        single = ops.block_grad_gemm(xd[id(a)], d.cuda(), ops.make_block_rc(idx, "cuda"), block, out_dtype=torch.float32)
        assert (got[o:o + n] - single.cpu().double().reshape(-1)).abs().max().item() <= 3e-5 * scale
    # bf16 sink, overwrite mode, second flush reuses the object
    sink = torch.empty(total * block * block, device="cuda", dtype=torch.bfloat16)
    off = 0
    for a, d, idx in problems:
        n = len(idx) * block * block
        batch.add(xd[id(a)], d.cuda(), idx, sink[off:off + n].view(-1, block), block)
        off += n
    batch.flush(accumulate=False)
    assert (sink.cpu().double() - truth).abs().max().item() <= 2 ** -7 * scale


def test_grouped_gemm_large_group_no_split(ops):
    """A group big enough to need no split-K (>= 148 tiles): whole-block tiles, direct epilogue."""
    torch.manual_seed(0)
    T, b = 512, 256
    xs = [torch.randn(T, 1024, device="cuda").bfloat16() for _ in range(4)]
    dys = [torch.randn(T, 2560, device="cuda").bfloat16() for _ in range(4)]
    idx = [(r, c) for r in range(10) for c in range(4)]               # every block of a 2560 x 1024 weight
    out = torch.zeros(4 * len(idx) * b * b, device="cuda")
    batch = ops.BlockGradBatch()
    for i in range(4):
        batch.add(xs[i], dys[i], idx, out[i * len(idx) * b * b:(i + 1) * len(idx) * b * b].view(-1, b), b)
    batch.flush(accumulate=False)
    for i in range(4):
        ref = dys[i].float().t() @ xs[i].float()                      # the full dense dW^T: every block is a slice of it
        got = out[i * len(idx) * b * b:(i + 1) * len(idx) * b * b].view(len(idx), b, b)
        want = torch.stack([ref[r * b:(r + 1) * b, c * b:(c + 1) * b] for r, c in idx])
        assert (got - want).abs().max().item() <= 2e-5 * want.abs().max().item()


@pytest.mark.parametrize("out_dtype,accumulate", [(torch.float32, False), (torch.bfloat16, True)])
def test_grouped_gemm_2sm_cta_pairs(ops, monkeypatch, out_dtype, accumulate):
    """cta_group::2 kernel (the default for large grouped b = 256 launches; SMT_GEMM_2SM=0 = single-CTA kernel): two
    blocks per SM pair, x operand split across the pair, dy strip loaded once when the two blocks share their block
    row.  Row-sharing pairs, unrelated pairs, an odd tail and a ragged token count; must match the single-CTA kernel
    (same K order => bit-identical) and the dense reference."""
    torch.manual_seed(11)
    T, b = 1000, 256                                                    # 1000 = 15 full 64-token stages + 40
    P = 5
    xs = [torch.randn(T, 1536, device="cuda").bfloat16() for _ in range(P)]
    dys = [torch.randn(T, 2048, device="cuda").bfloat16() for _ in range(P)]
    idx = [(0, 4)] + [(1, c) for c in (0, 5)] + [(2, c) for c in (1, 2, 3)] + [(3, c) for c in (0, 1, 2, 4, 5)] + \
          [(r, c) for r in (4, 5, 6, 7) for c in range(6)] + [(0, 1), (2, 5), (5, 0)]
    idx = list(dict.fromkeys(idx))
    uses = [idx[:-2]] + [idx] * (P - 1)                                 # odd total => one cluster with a single block
    offs = [0]
    for u in uses:
        offs.append(offs[-1] + len(u) * b * b)
    assert offs[-1] // (b * b) >= 148 and (offs[-1] // (b * b)) % 2 == 1
    init = (torch.randn(offs[-1], device="cuda") * 3).to(out_dtype)

    def run():
        out = init.clone() if accumulate else torch.zeros(offs[-1], device="cuda", dtype=out_dtype)
        batch = ops.BlockGradBatch()
        for i in range(P):
            batch.add(xs[i], dys[i], uses[i], out[offs[i]:offs[i + 1]].view(-1, b), b)
        launches0 = ops.LAUNCHES["total"]
        batch.flush(accumulate=accumulate)
        return out, ops.LAUNCHES["total"] - launches0

    monkeypatch.setenv("SMT_GEMM_2SM", "0")
    single, _ = run()
    monkeypatch.delenv("SMT_GEMM_2SM", raising=False)              # default: cta_group::2
    paired, launches = run()
    assert launches == 1 and ops.LAST_GROUP["cta_group_2"] and ops.LAST_GROUP["row_sharing_pairs"] > 40
    assert torch.equal(paired, single)
    for i in range(P):
        ref = dys[i].float().t() @ xs[i].float()
        got = paired[offs[i]:offs[i + 1]].view(len(uses[i]), b, b).float()
        want = torch.stack([ref[r * b:(r + 1) * b, c * b:(c + 1) * b] for r, c in uses[i]])
        if accumulate:
            want = want + init[offs[i]:offs[i + 1]].view(len(uses[i]), b, b).float()
        tol = 2e-5 if out_dtype == torch.float32 else 2 ** -7
        assert (got - want).abs().max().item() <= tol * want.abs().max().item()


@pytest.mark.parametrize("two_sm", [True, False])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_grouped_gemm_item_overwrite_flags_and_sq_partials(ops, monkeypatch, two_sm, out_dtype):
    """Work-item v2: (a) a problem added with accumulate=False OVERWRITES its blocks inside an accumulating launch (the
    lazy zero_grad of SMTAdam), the others accumulate; (b) the epilogue's per-block sums of squares describe exactly
    what is stored (after accumulation and rounding), are bit-reproducible, and differ between the cta_group::2 and the
    single-CTA kernel by fp32 summation order only."""
    torch.manual_seed(21)
    T, b, P = 448, 256, 4                                             # T < 512 => no split-K => the launch emits sums
    xs = [torch.randn(T, 1536, device="cuda").bfloat16() for _ in range(P)]
    dys = [torch.randn(T, 2560, device="cuda").bfloat16() for _ in range(P)]
    idx = [(r, c) for r in range(10) for c in range(6)][:-7] + [(9, 5)]             # 54 blocks, pairs + singles
    nblk = len(idx)
    n = nblk * b * b
    init = (torch.randn(P * n, device="cuda") * 50).to(out_dtype)
    overwrite = [True, False, True, False]
    if not two_sm:
        monkeypatch.setenv("SMT_GEMM_2SM", "0")

    def run():
        out = init.clone()
        sq = torch.full((2 * P * nblk,), -1.0, device="cuda")
        batch = ops.BlockGradBatch()
        for i in range(P):
            batch.add(xs[i], dys[i], idx, out[i * n:(i + 1) * n].view(-1, b), b, accumulate=not overwrite[i],
                      sq=sq, sq_slot0=2 * i * nblk)
        batch.flush(accumulate=True)
        return out, sq

    out, sq = run()
    assert ops.LAST_GROUP["emits_sq"] and ops.LAST_GROUP["cta_group_2"] == two_sm
    tol = 2 ** -7 if out_dtype == torch.bfloat16 else 3e-5
    for i in range(P):
        ref = dys[i].float().t() @ xs[i].float()
        want = torch.stack([ref[r * b:(r + 1) * b, c * b:(c + 1) * b] for r, c in idx])
        if not overwrite[i]:
            want = want + init[i * n:(i + 1) * n].view(nblk, b, b).float()
        got = out[i * n:(i + 1) * n].view(nblk, b, b).float()
        assert (got - want).abs().max().item() <= tol * want.abs().max().item(), i
    stored = out.view(P * nblk, 2, (b // 2) * b).double()              # halves: rows [0,128) and [128,256) of each block
    want_sq = (stored ** 2).sum(-1).reshape(-1)
    assert torch.allclose(sq.double(), want_sq, rtol=1e-5, atol=0)
    out2, sq2 = run()
    assert torch.equal(out, out2) and torch.equal(sq, sq2)               # deterministic


@pytest.mark.parametrize("block", [64, 128])
def test_grouped_gemm_sq_partials_small_blocks(ops, block):
    """b = 64 / 128: one tile per block - slot 0 holds the block's whole sum of squares, slot 1 is written as 0."""
    torch.manual_seed(block)
    T = 256
    x = torch.randn(T, 1024, device="cuda").bfloat16()
    dy = torch.randn(T, 1024, device="cuda").bfloat16()
    nb = 1024 // block
    idx = [(r, c) for r in range(nb) for c in range(nb)]
    if len(idx) > 200:
        idx = idx[:200]
    out = torch.empty(len(idx) * block * block, device="cuda", dtype=torch.bfloat16)
    sq = torch.full((2 * len(idx),), -1.0, device="cuda")
    batch = ops.BlockGradBatch()
    batch.add(x, dy, idx, out.view(-1, block), block, accumulate=False, sq=sq, sq_slot0=0)
    batch.flush(accumulate=True)
    if not ops.LAST_GROUP["emits_sq"]:
        pytest.skip("planner chose split-K for this shape")
    want = (out.view(len(idx), -1).double() ** 2).sum(-1)
    assert torch.allclose(sq.view(-1, 2)[:, 0].double(), want, rtol=1e-5, atol=0)
    assert not sq.view(-1, 2)[:, 1].any()


def test_compact_adam_with_partial_sqnorms_bit_exact(ops):
    """The Adam kernel adds n partial sums of squares itself (fixed order: oracle.partial_sqnorm_total) before forming
    the clip coefficient; fp32 state stays bit-identical to the numpy restatement."""
    rng = np.random.RandomState(3)
    N = 64 * 64 * 5
    p = (rng.randn(N) * 0.02).astype(np.float32)
    m = np.zeros(N, np.float32)
    v = np.zeros(N, np.float32)
    dp, dm, dv = (torch.from_numpy(a.copy()).cuda() for a in (p, m, v))
    hp = dict(lr=3e-4, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.0)
    for step, n_part in ((1, 2), (2, 300), (3, 1738), (4, 256)):
        g = torch.from_numpy(rng.randn(N).astype(np.float32)).bfloat16()
        parts = (g.float().view(5, -1) ** 2).sum(-1)
        parts = (parts.repeat_interleave((n_part + 4) // 5)[:n_part] / ((n_part + 4) // 5)).contiguous()
        total = O.partial_sqnorm_total(parts.numpy())
        gscale = O.clip_coef(total, np.float32(0.25), np.float32(1.0))
        ops.compact_adam(dp, dm, dv, g.cuda(), step=step, grad_scale=0.25, sqnorm=parts.cuda(), max_norm=1.0, **hp)
        p, m, v = O.adamw_fused_step(p, m, v, g.float().numpy(), step=step, gscale=gscale, **hp)
        assert np.array_equal(dp.cpu().numpy(), p), f"master differs at step {step} ({n_part} partials)"
        assert np.array_equal(dm.cpu().numpy(), m) and np.array_equal(dv.cpu().numpy(), v)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("block", [64, 128, 256])
def test_block_grad_gemm_token_count_edges(ops, block, dtype):
    """Ragged token counts around every stage height in use (64 / 128 / 256 tokens) and around split-K boundaries:
    the last TMA box is zero-filled past T, so any T must give the dense result.  Single-problem and grouped entry
    points, fp32 output, tolerance = fp32 accumulation error."""
    torch.manual_seed(block)
    fin, fout = 512, 768
    g = torch.Generator().manual_seed(block)
    nb = (fout // block) * (fin // block)
    perm = torch.randperm(nb, generator=g)[:min(nb, 7)].tolist()
    idx = [(p // (fin // block), p % (fin // block)) for p in perm]
    rc = ops.make_block_rc(idx, "cuda")
    for T in (1, 15, 16, 17, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 513, 1023, 1025, 2047, 2049, 4095, 4097):
        x = torch.randn(T, fin, device="cuda").to(dtype)
        dy = torch.randn(T, fout, device="cuda").to(dtype)
        ref = dy.float().t() @ x.float()
        want = torch.cat([ref[r * block:(r + 1) * block, c * block:(c + 1) * block] for r, c in idx])
        scale = max(want.abs().max().item(), 1e-3)
        got = ops.block_grad_gemm(x, dy, rc, block, out_dtype=torch.float32)
        assert (got - want).abs().max().item() <= 2e-5 * scale, (T, "single")
        out = torch.zeros(len(idx) * block, block, device="cuda")
        batch = ops.BlockGradBatch()
        batch.add(x, dy, idx, out, block)
        batch.flush(accumulate=False)
        assert (out - want).abs().max().item() <= 2e-5 * scale, (T, "grouped")


def test_grouped_gemm_2sm_token_count_edges(ops):
    """The cta_group::2 kernel with ragged / tiny token counts (zero-filled last stage, a single stage, one token)."""
    torch.manual_seed(4)
    b, P = 256, 4
    idx = [(r, c) for r in range(5) for c in range(8)]                  # 40 blocks per problem, 160 items
    for T in (1, 63, 64, 65, 200, 257):
        xs = [torch.randn(T, 2048, device="cuda").bfloat16() for _ in range(P)]
        dys = [torch.randn(T, 1280, device="cuda").bfloat16() for _ in range(P)]
        out = torch.zeros(P * len(idx) * b * b, device="cuda")
        batch = ops.BlockGradBatch()
        for i in range(P):
            batch.add(xs[i], dys[i], idx, out[i * len(idx) * b * b:(i + 1) * len(idx) * b * b].view(-1, b), b)
        batch.flush(accumulate=False)
        assert ops.LAST_GROUP["cta_group_2"], T
        for i in range(P):
            ref = dys[i].float().t() @ xs[i].float()
            got = out[i * len(idx) * b * b:(i + 1) * len(idx) * b * b].view(len(idx), b, b)
            want = torch.stack([ref[r * b:(r + 1) * b, c * b:(c + 1) * b] for r, c in idx])
            assert (got - want).abs().max().item() <= 2e-5 * max(want.abs().max().item(), 1e-3), T


# ---- fused dense projections (dense side of linearZ: smt.py:366, 406) ------------------------------------------------

@pytest.mark.parametrize("T,K,Ns,dtype", [
    (1000, 512, [512, 256, 256], torch.bfloat16),          # ragged T, GQA-shaped q/k/v
    (256, 1024, [256], torch.bfloat16),                    # one module, one tile
    (2309, 1536, [1024, 256], torch.float16),              # two modules, f16, ragged T
    (8192, 4096, [4096, 1024, 1024], torch.bfloat16),      # LLaMA-3-8B q/k/v at the bench's token count
])
def test_fused_linear_forward_vs_fp32(ops, T, K, Ns, dtype):
    """ONE tcgen05 launch for every module that reads x: each y_j must equal x @ W_j^T (fp32 accumulation, one rounding)
    - within half an ulp of the output type at the tensor's largest element plus the fp32 accumulation error."""
    torch.manual_seed(T + K)
    x = torch.randn(T, K, device="cuda").to(dtype)
    ws = [(torch.randn(n, K, device="cuda") * 0.05).to(dtype) for n in Ns]
    assert ops.fused_linear_supported(ws)
    ys = ops.fused_linear_forward(x, ws)
    eps = 2 ** -8 if dtype == torch.bfloat16 else 2 ** -11
    for y, w in zip(ys, ws):
        ref = x.float() @ w.float().t()
        assert y.shape == ref.shape and y.dtype == dtype
        assert (y.float() - ref).abs().max().item() <= (eps + 1e-4) * ref.abs().max().item()
        lib = torch.matmul(x, w.t()).float()                                   # the library GEMM it replaces
        assert (y.float() - ref).abs().max().item() <= 1.5 * (lib - ref).abs().max().item() + 1e-6
    ys2 = ops.fused_linear_forward(x, ws)
    assert all(torch.equal(a, b) for a, b in zip(ys, ys2))                    # deterministic


@pytest.mark.parametrize("T,K,Ns,dtype", [
    (1000, 512, [512, 256, 256], torch.bfloat16),
    (300, 192, [320, 64], torch.bfloat16),                 # dx narrower than one N tile, reduction lengths not x 256
    (2309, 1536, [1024, 256], torch.float16),
    (8192, 4096, [4096, 1024, 1024], torch.bfloat16),
])
def test_fused_linear_dgrad_vs_fp32(ops, T, K, Ns, dtype):
    """dx = sum_j dy_j @ W_j in ONE launch: the reduction runs through all (dy_j, W_j) pairs into one fp32 accumulator
    (the reference adds three separately rounded bf16 results)."""
    torch.manual_seed(T + K + 1)
    ws = [(torch.randn(n, K, device="cuda") * 0.05).to(dtype) for n in Ns]
    dys = [torch.randn(T, n, device="cuda").to(dtype) for n in Ns]
    assert ops.fused_linear_supported(ws, dgrad=True)
    dx = ops.fused_linear_dgrad(dys, ws)
    ref = sum(dy.float() @ w.float() for dy, w in zip(dys, ws))
    eps = 2 ** -8 if dtype == torch.bfloat16 else 2 ** -11
    assert dx.shape == (T, K) and dx.dtype == dtype
    err = (dx.float() - ref).abs().max().item()
    assert err <= (eps + 1e-4) * ref.abs().max().item()
    lib = sum(torch.matmul(dy, w) for dy, w in zip(dys, ws)).float()           # three library GEMMs + two bf16 adds
    assert err <= 1.05 * (lib - ref).abs().max().item() + 1e-6                 # one rounding instead of five
    assert torch.equal(dx, ops.fused_linear_dgrad(dys, ws))


def test_fused_linear_rejects_unsupported_shapes(ops):
    w_ok = torch.zeros(256, 512, device="cuda", dtype=torch.bfloat16)
    assert ops.fused_linear_supported([w_ok])
    assert not ops.fused_linear_supported([torch.zeros(128, 512, device="cuda", dtype=torch.bfloat16)])       # N % 256
    assert ops.fused_linear_supported([torch.zeros(128, 512, device="cuda", dtype=torch.bfloat16)], dgrad=True)
    assert not ops.fused_linear_supported([torch.zeros(256, 520, device="cuda", dtype=torch.bfloat16)])       # K % 64
    assert not ops.fused_linear_supported([w_ok.float()])                                                      # fp32
    assert not ops.fused_linear_supported([w_ok] * 4)
    assert not ops.fused_linear_supported([w_ok, torch.zeros(256, 1024, device="cuda", dtype=torch.bfloat16)])


# ---- strip-sharing run tiles ---------------------------------------------------------------------------------------------

def _run_patterns(block):
    nb = 1024 // block
    full_rows = [(r, c) for r in (1, 2) for c in range(nb)]                      # clustered: whole block rows
    mixed = [(0, 3), (0, 1), (3, 0), (0, 0), (2, 2), (0, 2), (3, 3), (1, 1), (3, 1), (0, nb - 1)][:max(4, nb)]
    mixed = list(dict.fromkeys((r % nb, c % nb) for r, c in mixed))
    return {"full_rows": full_rows, "mixed_unsorted": mixed, "single": [(nb - 1, nb - 1)]}


@pytest.mark.parametrize("T", [1000, 4096])
@pytest.mark.parametrize("block", [64, 128, 256])
def test_block_grad_gemm_run_launcher_vs_truth_and_block_tiles(ops, block, T):
    """Strip-sharing kernel through its private launcher (a tile = one block row x up to 4 / 2 of its blocks,
    b = 64 / 128): against fp64 truth and against the plain one-tile-per-block launcher, for whole block rows, an
    unsorted mixed list (runs + singles, output order = list order) and a single block; ragged token counts; bf16 and
    fp32 outputs; accumulate.  Then the automatic choice of the public op between the two kernels, for every block
    size."""
    torch.manual_seed(block + T)
    x = torch.randn(T, 1024).bfloat16()
    dy = torch.randn(T, 1024).bfloat16()
    xd, dyd = x.cuda(), dy.cuda()
    patterns = _run_patterns(block) if block != 256 else {}                        # b = 256 has no run tiles
    for name, idx in patterns.items():
        rc = ops.make_block_rc(idx, "cuda")
        runs = ops._runs_for(idx, block, xd.device)
        truth = O.block_grad_truth(x.reshape(1, T, -1), dy.reshape(1, T, -1), idx, block)
        scale = truth.abs().max().item()

        def out(dtype):
            return torch.empty((len(idx) * block, block), dtype=dtype, device="cuda")

        got32 = ops._gemm_runs(xd, dyd, runs, block, out(torch.float32), False)
        assert ops.LAST_SINGLE["kernel"] == "runs", name
        assert (got32.cpu().double() - truth).abs().max().item() <= 3e-5 * scale, name
        got16 = ops._gemm_runs(xd, dyd, runs, block, out(torch.bfloat16), False)
        assert (got16.cpu().double() - truth).abs().max().item() <= 2 ** -7 * scale, name
        assert torch.equal(got32, ops._gemm_runs(xd, dyd, runs, block, out(torch.float32), False))
        base = torch.randn_like(got32)
        acc = base.clone()
        ops._gemm_runs(xd, dyd, runs, block, acc, True)
        assert (acc - base - got32).abs().max().item() <= 3e-5 * scale, name
        plain = ops._gemm_blocks(xd, dyd, rc, block, out(torch.float32), False)
        assert ops.LAST_SINGLE["kernel"] == "blocks"
        assert (got32 - plain).abs().max().item() <= 3e-5 * scale, name           # different split points, same math
    # automatic choice: a big launch of wide runs => run tiles (b = 64 / 128); scattered singles / small launches => blocks
    nb = 1024 // block
    everything = [(r, c) for r in range(nb) for c in range(nb)]
    ops.block_grad_gemm(xd, dyd, ops.make_block_rc(everything, "cuda"), block, index_list=everything)
    assert ops.LAST_SINGLE["kernel"] == ("runs" if block == 64 else "blocks")     # 256 / 64 / 16 blocks: only b = 64 is big
    diag = [(i, i) for i in range(min(4, 1024 // block))]
    ops.block_grad_gemm(xd, dyd, ops.make_block_rc(diag, "cuda"), block, index_list=diag)
    assert ops.LAST_SINGLE["kernel"] == "blocks"


def test_block_grad_gemm_runs_many_tiles_no_split(ops):
    """More run tiles than SMs: several waves, no split-K, direct epilogue (b = 64, every block of a 2048 x 2048 weight)."""
    torch.manual_seed(5)
    T, b = 512, 64
    x = torch.randn(T, 2048, device="cuda").bfloat16()
    dy = torch.randn(T, 2048, device="cuda").bfloat16()
    idx = [(r, c) for r in range(32) for c in range(32)]
    out = torch.empty((len(idx) * b, b), dtype=torch.float32, device="cuda")
    got = ops._gemm_runs(x, dy, ops._runs_for(idx, b, x.device), b, out, False)
    assert ops.LAST_SINGLE["kernel"] == "runs" and ops.LAST_SINGLE["runs"] == 256
    ref = dy.float().t() @ x.float()
    want = torch.stack([ref[r * b:(r + 1) * b, c * b:(c + 1) * b] for r, c in idx]).reshape(-1, b)
    assert (got - want).abs().max().item() <= 2e-5 * want.abs().max().item()
