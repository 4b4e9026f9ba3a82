"""Edge tests of the kernels that make SMT: warm-up scoring, top-k selection, block / column movement and the compact
Adam step, at the sizes, dtypes, strides and values where a kernel goes wrong.

Every kernel here has an exact reference, so the bars are exact where the arithmetic allows it:
- elementwise fp32 additions (score_accumulate, act_score_accumulate) are replayed on the CPU in the kernel's order
  and must match bit for bit;
- top-k order is a Python sort on (score, rank), block and column movement is a byte copy;
- the fp32 Adam state must equal oracle.adamw_fused_step bit for bit, and its 16-bit outputs the RNE rounding of it.
Reductions whose order is not replayed are held, per block or per channel, to |got - ref64| <= c * 2^-24 * sum|terms|,
where c is the depth of the kernel's addition tree (plus one for gamma_c's 1 / (1 - c u) and one per extra rounding).
Thresholds that depend on the grid come from the device's SM count.  Every case runs twice and must be bit-identical to
itself.  The largest error-to-bound ratio of each bounded check is printed (run with -s to see it)."""
import math

import numpy as np
import pytest
import torch

from oracle import smt_oracle as O

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                       # unit roundoff of fp32
STRATEGIES = ("mean_abs", "abs_mean", "L1", "L2")
DTYPES = (torch.float32, torch.bfloat16, torch.float16)
INT_VIEW = {1: torch.uint8, 2: torch.int16, 4: torch.int32}


@pytest.fixture(scope="module")
def ops(built_library):
    from sparse_matrix_tuning_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bits(t: torch.Tensor) -> torch.Tensor:
    t = t.detach().cpu().contiguous()
    return t.view(INT_VIEW[t.element_size()])


def _same(got: torch.Tensor, want: torch.Tensor, what=""):
    """Bit-identical, except that any NaN matches any NaN (the GPU returns the canonical NaN, the CPU propagates the
    payload of its input)."""
    got, want = got.detach().cpu().contiguous(), want.detach().cpu().contiguous()
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    if got.dtype.is_floating_point:
        gn, wn = torch.isnan(got), torch.isnan(want)
        assert torch.equal(gn, wn), (what, "NaN positions", gn.nonzero()[:5].tolist(), wn.nonzero()[:5].tolist())
        got, want = got[~gn], want[~wn]
    bad = (_bits(got) != _bits(want)).nonzero()
    assert bad.numel() == 0, (what, bad.shape[0], bad[:5].reshape(-1).tolist(),
                              got.reshape(-1)[bad[:5, 0]].tolist(), want.reshape(-1)[bad[:5, 0]].tolist())


def _np_same(got: np.ndarray, want: np.ndarray, what=""):
    _same(torch.from_numpy(np.ascontiguousarray(got)), torch.from_numpy(np.ascontiguousarray(want)), what)


def _random_bits(shape, dtype, gen):
    """Random bit patterns of `dtype` (NaNs, infinities and subnormals included)."""
    es = torch.empty((), dtype=dtype).element_size()
    ib = INT_VIEW[es]
    lo, hi = (-2 ** 15, 2 ** 15) if es == 2 else (-2 ** 31, 2 ** 31)
    return torch.randint(lo, hi, shape, generator=gen, dtype=torch.int64).to(ib).view(dtype)


def _report(name, ratios):
    worst = max(ratios) if ratios else 0.0
    print(f"\n[bound ratio] {name}: {worst:.3g}")
    assert worst <= 1.0, (name, worst)


# ---- score_accumulate --------------------------------------------------------------------------------------------------

def _score_sizes(sms):
    """n in {1, 7, 8, 9}, and around one and two grid strides of the vector kernel: its grid is
    min(ceil(n / 8 / 256), 4 * SMs) CTAs of 256 threads, each taking 8-element groups, so one stride covers
    8 * 256 * 4 * SMs elements; thread 0 enters the unrolled main loop only when n exceeds it."""
    stride = 8 * 256 * 4 * sms
    sizes = [1, 7, 8, 9]
    for k in (1, 2):
        for base in (k * stride - 8, k * stride + 8):
            sizes += [base, base + 8, base + 3]
    return sizes


@pytest.mark.parametrize("dtype", DTYPES)
def test_score_accumulate_grid_strides_and_scalar_path(ops, sms, dtype):
    """acc += grad.float(): one fp32 addition per element, so the result is exact whatever the grid.  Views offset by
    one element are not 16-byte aligned and take the scalar kernel for the whole call."""
    gen = torch.Generator().manual_seed(11)
    for n in _score_sizes(sms):
        for offset in (0, 1):
            acc0 = torch.randn(n + offset, generator=gen)
            grad = (torch.randn(n + offset, generator=gen) * 4).to(dtype)
            for i, (a, g) in zip((offset, n // 2 + offset, n + offset - 1, n // 3 + offset),
                                 ((float("inf"), float("-inf")), (float("nan"), 1.0), (2.0, float("nan")),
                                  (1.0, float("inf")))):
                acc0[i] = a
                grad[i] = g
            want = acc0[offset:] + grad[offset:].float()
            gd = grad.cuda()
            runs = []
            for _ in range(2):
                acc = acc0.cuda()
                ops.score_accumulate(acc[offset:], gd[offset:])
                runs.append(acc[offset:].cpu())
            _same(runs[0], want, (n, offset))
            assert torch.equal(_bits(runs[0]), _bits(runs[1])), (n, offset)


def test_score_accumulate_and_sqnorm_accept_empty_tensors(ops):
    """An empty CUDA tensor has data_ptr() == 0; n = 0 must need no data pointer.  grad_sqnorm still writes 0."""
    for dtype in DTYPES:
        acc = torch.empty(0, device="cuda")
        ops.score_accumulate(acc, torch.empty(0, device="cuda", dtype=dtype))
        out = torch.full((1,), 7.0, device="cuda")
        ops.grad_sqnorm(torch.empty(0, device="cuda", dtype=dtype), out=out)
        assert out.item() == 0.0


# ---- block sums and block score reduction ------------------------------------------------------------------------------

def _partial_depth(block, dtype):
    """Depth of the addition tree of block_partial + block_sum for one term: the pair(s) of a 128-bit load, one
    addition per pass into s0 / s1, s0 + s1, then 5 warp and 5 block butterfly levels."""
    vec = 4 if dtype == torch.float32 else 8
    passes = block * block // (256 * vec)
    pair_levels = 1 if dtype == torch.float32 else 2
    return pair_levels + passes + 1 + 10


def _blocked_view(rb, cb, block, dtype, gen, const_blocks=()):
    """A [rb*b, cb*b] view with ld > cols and a 16-byte aligned, non-zero storage offset, whose blocks have
    magnitudes spread over 12 binades; `const_blocks` = [(r, c, value)] are filled with one value."""
    es = torch.empty((), dtype=dtype).element_size()
    a = 16 // es                                          # elements per 16 bytes
    R, C = rb * block, cb * block
    base = torch.full((R + 3, C + 5 * a), float("nan"), dtype=torch.float32)
    scale = 2.0 ** torch.randint(-6, 7, (rb, cb), generator=gen).float()
    vals = torch.randn(R, C, generator=gen) * scale.repeat_interleave(block, 0).repeat_interleave(block, 1)
    for r, c, v in const_blocks:
        vals[r * block:(r + 1) * block, c * block:(c + 1) * block] = v
    base[2:2 + R, 3 * a:3 * a + C] = vals
    dev = base.to(dtype).cuda()
    view = dev[2:2 + R, 3 * a:3 * a + C]
    assert view.stride(0) > C and view.storage_offset() > 0 and view.data_ptr() % 16 == 0
    return view


def _blocks64(x: torch.Tensor, block: int) -> torch.Tensor:
    R, C = x.shape
    return x.double().cpu().reshape(R // block, block, C // block, block)


CONST = ((0, 1, 8.0), (1, 0, -0.03125), (2, 4, 2.0 ** -9))   # power-of-two constant blocks: exact results


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("block", [64, 128, 256])
def test_block_sum_accumulate_and_finalize_per_block(ops, block, dtype):
    gen = torch.Generator().manual_seed(block + len(str(dtype)))
    rb, cb = 3, 5
    g1 = _blocked_view(rb, cb, block, dtype, gen, CONST)
    g2 = _blocked_view(rb, cb, block, dtype, gen)
    depth = _partial_depth(block, dtype)
    ratios = []
    runs = []
    for _ in range(2):
        sums = torch.zeros(rb, cb, device="cuda")
        ops.block_sum_accumulate(sums, g1, block)
        first = sums.clone()
        ops.block_sum_accumulate(sums, g2, block)
        runs.append((first.cpu(), sums.cpu()))
    assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(runs[0], runs[1]))
    first, second = runs[0]
    b1, b2 = _blocks64(g1, block), _blocks64(g2, block)
    ref1, abs1 = b1.sum((1, 3)), b1.abs().sum((1, 3))
    ref2, abs2 = ref1 + b2.sum((1, 3)), abs1 + b2.abs().sum((1, 3))
    c1 = depth + 1                                        # + 1: gamma's 1 / (1 - c u)
    c2 = depth + 2                                        # + the addition into the existing sums
    ratios += ((first.double() - ref1).abs() / (c1 * U * abs1)).reshape(-1).tolist()
    ratios += ((second.double() - ref2).abs() / (c2 * U * abs2)).reshape(-1).tolist()
    for r, c, v in CONST:
        assert first[r, c].item() == v * block * block, (r, c)
    _report(f"block_sum_accumulate b={block} {dtype} (c = {c1} / {c2})", ratios)
    # finalize: |sums| / b^2, b^2 a power of two: exact
    sums = runs[0][1].cuda()
    got = ops.block_sum_finalize(sums, block).cpu()
    assert torch.equal(_bits(got), _bits((sums.cpu() / float(block * block)).abs()))
    fin1 = ops.block_sum_finalize(first.cuda(), block).cpu()
    for r, c, v in CONST:
        assert fin1[r, c].item() == abs(v), (r, c)


@pytest.mark.parametrize("strategy", STRATEGIES)
@pytest.mark.parametrize("block", [64, 128, 256])
def test_block_score_reduce_per_block_bounds(ops, block, strategy):
    """Per-block bounds: a block 2^12 times smaller than its neighbours is held to its own terms, not the tensor's."""
    gen = torch.Generator().manual_seed(block * 7 + len(strategy))
    rb, cb = 4, 3
    acc = _blocked_view(rb, cb, block, torch.float32, gen, ((0, 1, 8.0), (3, 2, -0.03125), (2, 0, 2.0 ** -9)))
    got = ops.block_score_reduce(acc, block, strategy).cpu()
    assert torch.equal(_bits(got), _bits(ops.block_score_reduce(acc, block, strategy).cpu()))
    b = _blocks64(acc, block)
    depth = _partial_depth(block, torch.float32)
    cnt = float(block * block)
    if strategy == "L2":
        # bound the square: one rounding per product, the tree, and the root (|got^2 - s| <= 2u s + ...)
        c = depth + 1 + 2 + 1
        ref, scale = (b * b).sum((1, 3)), (b * b).sum((1, 3))
        err = (got.double() ** 2 - ref).abs()
    else:
        c = depth + 1
        terms = b if strategy == "mean_abs" else b.abs()
        ref, scale = terms.sum((1, 3)), b.abs().sum((1, 3))
        div = 1.0 if strategy == "L1" else cnt
        if strategy == "mean_abs":
            ref = ref.abs()
        err = (got.double() * div - ref).abs()          # the division by b^2 is exact
    _report(f"block_score_reduce b={block} {strategy} (c = {c})", (err / (c * U * scale)).reshape(-1).tolist())
    for r, cc, v in ((0, 1, 8.0), (3, 2, -0.03125), (2, 0, 2.0 ** -9)):
        want = {"mean_abs": abs(v), "abs_mean": abs(v), "L1": abs(v) * cnt, "L2": abs(v) * block}[strategy]
        assert got[r, cc].item() == want, (r, cc, got[r, cc].item(), want)


# ---- activation (channel) scoring ------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES)
def test_act_score_accumulate_bit_exact_and_channel_reduce_bounds(ops, dtype):
    """acc[S, C] += sum_b |x[b]|: the kernel forms the batch sum from 0 in batch order, then adds it to acc; the CPU
    replays that order bit for bit.  channel_score_reduce: 8 row lanes each add every 8th row in order, then the 8
    lane sums are added in order, so a term passes through at most ceil(S / 8) + 7 additions."""
    gen = torch.Generator().manual_seed(len(str(dtype)))
    ratios = {s: [] for s in STRATEGIES}
    for batch in (1, 3):
        for seq in (1, 7, 8, 9, 513):
            for ch in (8, 128, 136, 4104):
                x = (torch.randn(batch, seq, ch, generator=gen) * 2.0 ** torch.randint(-8, 9, (1, 1, ch), generator=gen)
                     ).to(dtype)
                acc0 = torch.rand(seq, ch, generator=gen)
                s = torch.zeros(seq, ch)
                for b in range(batch):
                    s = s + x[b].float().abs()
                want = acc0 + s
                xd = x.cuda()
                runs = []
                for _ in range(2):
                    acc = acc0.cuda()
                    ops.act_score_accumulate(acc, xd)
                    runs.append(acc)
                assert torch.equal(_bits(runs[0]), _bits(want)), (batch, seq, ch)
                assert torch.equal(runs[0], runs[1])
                if dtype == torch.bfloat16:                # the reduce reads fp32 only: once per shape is enough
                    _channel_reduce_check(ops, runs[0], ratios)
    if dtype == torch.bfloat16:
        for s in STRATEGIES:
            _report(f"channel_score_reduce {s}", ratios[s])


def _channel_reduce_check(ops, acc, ratios):
    seq = acc.shape[0]
    a = acc.double().cpu()
    depth = -(-seq // 8) + 7
    for s in STRATEGIES:
        got = ops.channel_score_reduce(acc, s)
        assert torch.equal(got, ops.channel_score_reduce(acc, s))
        got = got.cpu().double()
        l1 = a.abs().sum(0)
        if s == "L2":
            c = depth + 1 + 1 + 2
            err, scale = (got ** 2 - (a * a).sum(0)).abs(), (a * a).sum(0)
        elif s == "L1":
            c = depth + 1
            err, scale = (got - l1).abs(), l1
        else:                                               # one more rounding: the division by S
            c = depth + 2
            ref = l1 / seq if s == "mean_abs" else (a.sum(0) / seq).abs()
            err, scale = (got - ref).abs(), l1 / seq
        ratios[s] += (err / (c * U * scale.clamp_min(1e-300))).tolist()


def test_channel_score_reduce_direct_small_widths(ops):
    """Direct calls with 4 and 12 channels (one CTA mostly idle) and signed inputs, where abs_mean and mean_abs
    differ."""
    gen = torch.Generator().manual_seed(5)
    ratios = {s: [] for s in STRATEGIES}
    for ch in (4, 12):
        for seq in (1, 7, 8, 9, 513):
            acc = torch.randn(seq, ch, generator=gen).cuda()
            _channel_reduce_check(ops, acc, ratios)
    for s in STRATEGIES:
        _report(f"channel_score_reduce direct {s}", ratios[s])


# ---- top-k ---------------------------------------------------------------------------------------------------------------

F32_MAX = float(np.finfo(np.float32).max)
_ONE_UP = float(np.nextafter(np.float32(1), np.float32(2)))
_POOL = np.array([0.0, -0.0, 1e-45, -1e-45, 1.4e-40, -1.4e-40, float("inf"), float("-inf"), F32_MAX, -F32_MAX,
                  1.0, _ONE_UP, float(np.nextafter(np.float32(1), np.float32(0))),
                  float(np.nextafter(np.float32(_ONE_UP), np.float32(2))), 0.5, -0.5], dtype=np.float32)


def _topk_scores(n, kind, rng):
    if kind == "equal":
        return np.full(n, 0.75, np.float32)
    s = _POOL[rng.randint(len(_POOL), size=n)]
    fresh = rng.rand(n) < 0.3
    s[fresh] = rng.randn(int(fresh.sum())).astype(np.float32)
    return s


def _ranks(n, mode, rng):
    """(rank for the kernel or None, rank used by the reference order)."""
    if mode == "null":
        return None, np.arange(n)
    rank = rng.permutation(n) if mode == "perm" else n - 1 - np.arange(n)
    return rank, rank


def _ref_order(s, r, lo, hi):
    """Descending (score, rank) over [lo, hi) of the Python lists s, r: the order of the reference's tuples, with
    -0.0 taken as 0.0."""
    return sorted(range(lo, hi), key=lambda i: (s[i] + 0.0, r[i]), reverse=True)


def _run_topk(ops, scores, rank, offs, ks):
    sd = torch.from_numpy(scores).cuda()
    if rank is None:
        args = ()
    else:
        inv = np.empty_like(rank)
        inv[rank] = np.arange(len(rank))
        args = (torch.from_numpy(rank.astype(np.int32)).cuda(), torch.from_numpy(inv.astype(np.int32)).cuda())
    idx, oo = ops.topk_blocks(sd, offs, ks, *args)
    idx2, _ = ops.topk_blocks(sd, offs, ks, *args)
    assert torch.equal(idx, idx2)
    return idx.cpu().tolist(), oo


@pytest.mark.parametrize("kind", ["mixed", "equal"])
@pytest.mark.parametrize("mode", ["null", "perm", "reversed"])
def test_topk_single_segment_around_shared_memory_limit(ops, kind, mode):
    """k on either side of the 8 192 keys that fit shared memory (beyond: a global-memory bitonic sort)."""
    rng = np.random.RandomState(len(kind) * 10 + len(mode))
    for n in (1, 8192, 8193, 16385, 98304):
        scores = _topk_scores(n, kind, rng)
        rank, ref_rank = _ranks(n, mode, rng)
        order = _ref_order(scores.tolist(), ref_rank.tolist(), 0, n)
        for k in (1, 2, 4096, 4097, 8191, 8192, 8193, 16384, n):
            got, oo = _run_topk(ops, scores, rank, [0, n], [k])
            assert oo == [0, min(k, n)]
            assert got == order[:k], (n, k)


@pytest.mark.parametrize("mode", ["null", "perm", "reversed"])
def test_topk_many_segments_shared_and_global(ops, mode):
    """One launch mixing shared- and global-memory segments.  The first three global segments are adjacent with
    k > len / 2: their workspace slices (2 * begin, 2 * len keys each) would overlap if they started at `begin`."""
    rng = np.random.RandomState(len(mode))
    segs = [(9000, 8500), (10000, 9000), (12000, 11000), (0, 5), (1, 1), (1, 0), (500, 1000), (8192, 8192),
            (20000, 8193), (3, 2), (16385, 16385), (100, 0), (7, 7), (0, 0), (8193, 4097), (40, 39)]
    offs = [0]
    for length, _ in segs:
        offs.append(offs[-1] + length)
    n = offs[-1]
    for kind in ("mixed", "equal"):
        scores = _topk_scores(n, kind, rng)
        rank, ref_rank = _ranks(n, mode, rng)
        got, oo = _run_topk(ops, scores, rank, offs, [k for _, k in segs])
        sl, rl = scores.tolist(), ref_rank.tolist()
        for s, (length, k) in enumerate(segs):
            want = _ref_order(sl, rl, offs[s], offs[s + 1])[:max(0, k)]
            assert got[oo[s]:oo[s + 1]] == want, (kind, s, length, k)


def test_topk_norm_dist_llama8b_b64(ops):
    """The `norm_dist` launch of LLaMA-3-8B with MLP at b = 64: 32 layers x (q, k, v, gate, up, down) = 192
    segments; gate / up / down have 14 336 blocks each, so k = 9 000 takes the global path there and the shared path
    (k = len) on q / k / v.  Scores with many ties, ranks = the reversed flat index norm_dist uses."""
    sizes = [4096, 1024, 1024, 14336, 14336, 14336] * 32
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    n = offs[-1]
    rng = np.random.RandomState(8)
    scores = (rng.randint(0, 2048, size=n) / 2048.0).astype(np.float32)
    rank = (n - 1 - np.arange(n)).astype(np.int64)
    got, oo = _run_topk(ops, scores, rank, offs, [9000] * len(sizes))
    sl, rl = scores.tolist(), rank.tolist()
    for s in range(len(sizes)):
        want = _ref_order(sl, rl, offs[s], offs[s + 1])[:9000]
        assert got[oo[s]:oo[s + 1]] == want, s


def test_topk_norm_dist_selection_matches_oracle(ops):
    """smt_helper's norm_dist selection against the oracle's per-matrix argsort on tie-free scores (two LLaMA-3-8B
    layers at b = 64, n = 9 000 per matrix)."""
    from sparse_matrix_tuning_b200.smt import smt_helper as H
    shapes = {"q_proj": (64, 64), "k_proj": (16, 64), "v_proj": (16, 64), "gate_proj": (224, 64),
              "up_proj": (224, 64), "down_proj": (64, 224)}
    keys = [(m, layer) for layer in (0, 1) for m in shapes]
    total = sum(shapes[m][0] * shapes[m][1] for m, _ in keys)
    vals = torch.from_numpy(np.random.RandomState(3).permutation(total).astype(np.float32) / total)
    scores, off = {}, 0
    for m, layer in keys:
        r, c = shapes[m]
        scores[(m, layer)] = vals[off:off + r * c].reshape(r, c)
        off += r * c
    want = O.select_from_scores(scores, 9000, "norm_dist")
    got = H.select_submatrix_from_scores(keys, [s.cuda() for s in scores.values()], 9000, "norm_dist")
    assert list(got.items()) == list(want.items())


# ---- block gather / scatter -------------------------------------------------------------------------------------------

def _weight_views(shapes, block, dtype, gen):
    """Weights [r*b, c*b] as views (ld > cols, 16-byte aligned non-zero offset) into buffers that hold a NaN bit
    pattern everywhere else; the weights themselves hold random bit patterns."""
    es = torch.empty((), dtype=dtype).element_size()
    a = 16 // es
    bufs, views = [], []
    for r, c in shapes:
        R, C = r * block, c * block
        buf = torch.full((R + 2, C + 3 * a), float("nan"), dtype=dtype)
        buf[1:1 + R, a:a + C] = _random_bits((R, C), dtype, gen)
        buf = buf.cuda()
        bufs.append(buf)
        views.append(buf[1:1 + R, a:a + C])
    return bufs, views


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("block", [64, 128, 256])
def test_block_gather_scatter_views_many_weights(ops, block, dtype):
    gen = torch.Generator().manual_seed(block + len(str(dtype)))
    bufs, views = _weight_views([(3, 5), (2, 1), (1, 4)], block, dtype, gen)
    entries = [(0, 2, 4), (1, 1, 0), (0, 0, 0), (2, 0, 3), (0, 2, 0), (1, 0, 0), (0, 1, 3), (2, 0, 1), (0, 0, 4)]
    _gather_scatter_check(ops, bufs, views, entries, block, dtype, gen)


def test_block_gather_scatter_3000_blocks(ops):
    gen = torch.Generator().manual_seed(3000)
    block = 64
    bufs, views = _weight_views([(60, 64), (5, 7)], block, torch.bfloat16, gen)
    perm = torch.randperm(60 * 64, generator=gen)[:2990].tolist()
    entries = [(0, p // 64, p % 64) for p in perm] + [(1, r, c) for r, c in ((4, 6), (0, 0), (4, 0), (0, 6), (2, 3))]
    order = torch.randperm(len(entries), generator=gen).tolist()
    _gather_scatter_check(ops, bufs, views, [entries[i] for i in order], block, torch.bfloat16, gen)


def _gather_scatter_check(ops, bufs, views, entries, block, dtype, gen):
    n = len(entries)
    tab = ops.make_block_table([(views[w], r, c) for w, r, c in entries], "cuda")
    host = [v.cpu() for v in views]
    want = torch.stack([host[w][r * block:(r + 1) * block, c * block:(c + 1) * block] for w, r, c in entries])
    for _ in range(2):
        comp = torch.full((n * block, block), 1.5, dtype=dtype, device="cuda")
        ops.block_gather(tab, n, block, comp)
        assert torch.equal(_bits(comp), _bits(want.reshape(n * block, block)))
    new = _random_bits((n * block, block), dtype, gen)
    expect = [b.cpu() for b in bufs]
    a = 16 // new.element_size()
    for i, (w, r, c) in enumerate(entries):
        expect[w][1 + r * block:1 + (r + 1) * block, a + c * block:a + (c + 1) * block] = new[i * block:(i + 1) * block]
    for _ in range(2):                                    # the second scatter writes the same bytes again
        ops.block_scatter(tab, n, block, new.cuda())
        for b, e in zip(bufs, expect):
            assert torch.equal(_bits(b), _bits(e))        # every byte outside the blocks unchanged


# ---- column / channel movement ------------------------------------------------------------------------------------------

def _channel_list(n, width, gen):
    """n distinct channels in random (unsorted) order; the last column always, the first one too when n >= 2."""
    if n == 1:
        return [width - 1]
    idx = [c for c in torch.randperm(width, generator=gen).tolist() if c not in (0, width - 1)][:n - 2]
    idx.insert(len(idx) // 3, width - 1)
    idx.insert(2 * len(idx) // 3, 0)
    return idx


@pytest.mark.parametrize("dtype", [torch.int16, torch.int32])
def test_column_gather_scatter_tile_edges(ops, dtype):
    """32 x 32 tiles: out_features and n on either side of a tile; unsorted channels including the first and last
    column; W a view with ldw > in_features and a non-zero offset in a buffer of sentinels."""
    gen = torch.Generator().manual_seed(dtype.itemsize)
    F = 1037
    for out_f in (8, 32, 40, 4104):
        for n in (1, 31, 32, 33, 1000):
            buf = torch.randint(-1000, 1000, (out_f, F + 11), generator=gen, dtype=torch.int32).to(dtype)
            idx = _channel_list(n, F, gen)
            bd = buf.cuda()
            W = bd[:, 3:3 + F]
            d_idx = torch.tensor(idx, dtype=torch.int32, device="cuda")
            for _ in range(2):
                comp = torch.full((n, out_f), -7, dtype=dtype, device="cuda")
                ops.column_gather(W, d_idx, comp)
                assert torch.equal(comp.cpu(), buf[:, 3:3 + F][:, idx].t()), (out_f, n)
            new = torch.randint(-1000, 1000, (n, out_f), generator=gen, dtype=torch.int32).to(dtype)
            expect = buf.clone()
            expect[:, [3 + i for i in idx]] = new.t()
            for _ in range(2):
                ops.column_scatter(W, d_idx, new.cuda())
                assert torch.equal(bd.cpu(), expect), (out_f, n)


@pytest.mark.parametrize("dtype", [torch.int16, torch.int32])
def test_channel_gather_padding_and_strides(ops, dtype):
    gen = torch.Generator().manual_seed(10 + dtype.itemsize)
    F = 777
    for T in (1, 1000):
        for n in (1, 31, 32, 33, 1000):
            buf = torch.randint(1, 1000, (T, F + 13), generator=gen, dtype=torch.int32).to(dtype)
            x = buf.cuda()[:, 5:5 + F]
            idx = _channel_list(min(n, F), F, gen) + [-1] * max(0, n - F)
            if n >= 4:
                for j in (1, n // 2, n - 1):
                    idx[j] = -1
            idx = [idx[i] for i in torch.randperm(n, generator=gen).tolist()] if n > 2 else idx
            want = torch.zeros(T, n, dtype=dtype)
            for i, c in enumerate(idx):
                if c >= 0:
                    want[:, i] = buf[:, 5 + c]
            d_idx = torch.tensor(idx, dtype=torch.int32, device="cuda")
            for _ in range(2):
                out = torch.full((T, n), -3, dtype=dtype, device="cuda")
                ops.channel_gather(x, d_idx, out)
                assert torch.equal(out.cpu(), want), (T, n)


# ---- grad_sqnorm ----------------------------------------------------------------------------------------------------------

SQ_SIZES = (1, 7, 8, 9, 8191, 8_388_600, 8_388_608, 3 * 8_388_608 + 5)


def _sqnorm_chain(n):
    """Longest addition chain a term of smt_grad_sqnorm passes through before the two block butterflies (5 + 5 levels
    each, the 20 of the bound): stage 1 takes grid = clamp(ceil(n/8 / 1024), 1, 1024) CTAs, CTA j owns
    ceil(n8 / grid) contiguous 8-vectors; its thread 0 owns c = ceil(per_cta / 256) of them, consumed 4 at a time
    (8-term chains, a 2-level pair tree, one addition to s) and then one by one (8 additions each); the last CTA adds
    the n % 8 tail, one element per thread.  Stage 2 thread 0 adds ceil(grid / 256) partials.  + 1 for the product's
    rounding, + 1 for gamma's 1 / (1 - c u)."""
    n8 = n // 8
    grid = max(1, min(1024, -(-n8 // 1024)))
    per = -(-n8 // grid) if n8 else 0
    c = -(-per // 256)
    main, rem = c // 4, c % 4
    stage1 = max(10 + main + 8 * rem if main else 0, 8 * rem) + (1 if n % 8 else 0)
    return stage1 + -(-grid // 256) + 2


@pytest.mark.parametrize("dtype", DTYPES)
def test_grad_sqnorm_partition_tail_and_offsets(ops, dtype):
    gen = torch.Generator().manual_seed(len(str(dtype)))
    es = torch.empty((), dtype=dtype).element_size()
    a = 16 // es
    ratios = []
    for n in SQ_SIZES:
        g = torch.randn(n, generator=gen).to(dtype)
        ref = float((g.double() ** 2).sum())
        gd = g.cuda()
        got = ops.grad_sqnorm(gd).item()
        assert ops.grad_sqnorm(gd).item() == got
        buf = torch.zeros(n + a, dtype=dtype, device="cuda")
        buf[a:] = gd
        assert ops.grad_sqnorm(buf[a:]).item() == got                 # same values, another 16-byte offset: same bits
        L = _sqnorm_chain(n)
        ratios.append(abs(got - ref) / ((L + 20) * U * ref))
    _report(f"grad_sqnorm {dtype}", ratios)
    for n in (9, 8191, 8_388_600):
        gd = torch.randn(n, generator=gen).to(dtype).cuda()
        for pos in (0, n // 2, n - 1):
            for val, check in ((float("inf"), math.isinf), (float("nan"), math.isnan)):
                h = gd.clone()
                h[pos] = val
                assert check(ops.grad_sqnorm(h).item()), (n, pos, val)


# ---- compact Adam -------------------------------------------------------------------------------------------------------

HP = dict(lr=3e-4, beta1=0.9, beta2=0.95, eps=1e-8)


def _state(n, rng):
    p = (rng.randn(n) * 0.02).astype(np.float32)
    m = (rng.randn(n) * 1e-3).astype(np.float32)
    v = (rng.rand(n) * 1e-6).astype(np.float32)
    return p, m, v


def _oracle_step(p, m, v, g, step, gscale, wd):
    with np.errstate(all="ignore"):
        return O.adamw_fused_step(p, m, v, g, step=step, gscale=gscale, weight_decay=wd, **HP)


def _gscale(total, grad_scale, max_norm):
    if total is None:
        return np.float32(grad_scale)
    with np.errstate(all="ignore"):
        return O.clip_coef(np.float32(total), np.float32(grad_scale), np.float32(max_norm))


def _block_weight(rb, cb, block, dtype, gen):
    """A weight view inside a buffer of sentinels (pad rows and columns)."""
    es = torch.empty((), dtype=dtype).element_size()
    a = 16 // es
    buf = torch.full((rb * block + 2, cb * block + 2 * a), -0.375, dtype=dtype)
    buf[1:1 + rb * block, a:a + cb * block] = torch.randn(rb * block, cb * block, generator=gen).to(dtype)
    buf = buf.cuda()
    return buf, buf[1:1 + rb * block, a:a + cb * block], (1, a)


def _run_adam_case(ops, n, gdt, cdt, wdt, gen, rng, *, block=64, blocks=None, rbcb=(3, 4), step=3, grad_scale=0.5,
                   wd=0.01, n_sq=3, max_norm=1.0, g=None):
    """One compact_adam call, twice from the same state, against the oracle; returns nothing, asserts everything."""
    if blocks is not None:
        n = len(blocks) * block * block
    p, m, v = _state(n, rng)
    if g is None:
        g = torch.from_numpy(rng.randn(n).astype(np.float32) * 0.05).to(gdt)
    gf = g.float().numpy()
    sq, total = None, None
    if n_sq:
        parts = (rng.rand(n_sq) * float((g.double() ** 2).sum()) * 2 / n_sq).astype(np.float32)
        sq, total = torch.from_numpy(parts), O.partial_sqnorm_total(parts)
    gscale = _gscale(total if max_norm > 0 else None, grad_scale, max_norm)
    wp, wm, wv = _oracle_step(p, m, v, gf, step, gscale, wd)
    kw = {}
    if wdt is not None:
        buf, W, (r0, c0) = _block_weight(*rbcb, block, wdt, gen)
        before = buf.cpu()
        kw = dict(table=ops.make_block_table([(W, r, c) for r, c in blocks], "cuda"), n_blocks=len(blocks),
                  block=block, w_dtype=wdt)
    results = []
    for _ in range(2):
        dp, dm, dv = (torch.from_numpy(x.copy()).cuda() for x in (p, m, v))
        comp = torch.full((n,), 3.0, dtype=cdt, device="cuda") if cdt is not None else None
        if wdt is not None:
            buf.copy_(before)
        ops.compact_adam(dp, dm, dv, g.cuda(), step=step, grad_scale=grad_scale,
                         sqnorm=sq.cuda() if sq is not None else None, max_norm=max_norm, compact_out=comp,
                         weight_decay=wd, **HP, **kw)
        what = (n, gdt, cdt, wdt, block, step, n_sq, max_norm)
        _np_same(dp.cpu().numpy(), wp, ("master",) + what)
        _np_same(dm.cpu().numpy(), wm, ("exp_avg",) + what)
        _np_same(dv.cpu().numpy(), wv, ("exp_avg_sq",) + what)
        master = torch.from_numpy(wp)
        if cdt is not None:
            _same(comp, master.to(cdt), ("compact",) + what)
        if wdt is not None:
            expect = before.clone()
            mb = master.to(wdt).reshape(len(blocks), block, block)
            for i, (r, c) in enumerate(blocks):
                expect[r0 + r * block:r0 + (r + 1) * block, c0 + c * block:c0 + (c + 1) * block] = mb[i]
            _same(buf, expect, ("W",) + what)
            results.append(buf.cpu())
        results.append(dp.cpu())
    half = len(results) // 2
    for a, b in zip(results[:half], results[half:]):
        assert torch.equal(_bits(a), _bits(b))


OPT_DTYPES = (None, torch.float32, torch.bfloat16, torch.float16)


@pytest.mark.parametrize("gdt", DTYPES)
def test_compact_adam_every_dtype_instantiation(ops, gdt):
    """Every (grad, compact_out, W) combination, W written back into a view with sentinels around the blocks, the
    blocks in the last block row and the last block column."""
    gen = torch.Generator().manual_seed(len(str(gdt)))
    rng = np.random.RandomState(len(str(gdt)))
    for cdt in OPT_DTYPES:
        for wdt in OPT_DTYPES:
            _run_adam_case(ops, 0, gdt, cdt, wdt, gen, rng, blocks=[(2, 3), (0, 0), (1, 2), (2, 0)])


@pytest.mark.parametrize("block,wdt", [(64, torch.bfloat16), (128, torch.float16), (256, torch.float32)])
def test_compact_adam_block_write_back_multi_pass(ops, sms, block, wdt):
    """More elements than one pass of the grid (SMs x 10 CTAs x 256 threads x 4 elements), written back into a random
    three quarters of a weight's blocks in random order."""
    gen = torch.Generator().manual_seed(block)
    rng = np.random.RandomState(block)
    n_blocks = -(-(sms * 10 * 256 * 4 + 1) // (block * block)) + 2
    cb = 8
    rb = -(-n_blocks * 4 // (3 * cb))
    perm = torch.randperm(rb * cb, generator=gen)[:n_blocks].tolist()
    blocks = [(p // cb, p % cb) for p in perm]
    if (rb - 1, cb - 1) not in blocks:
        blocks[0] = (rb - 1, cb - 1)
    _run_adam_case(ops, 0, torch.bfloat16, torch.bfloat16, wdt, gen, rng, block=block, blocks=blocks, rbcb=(rb, cb))


def test_compact_adam_sizes_and_clip_cases(ops, sms):
    gen = torch.Generator().manual_seed(1)
    rng = np.random.RandomState(1)
    for n in (8, 1032, sms * 10 * 256 * 4 + 8):
        _run_adam_case(ops, n, torch.float16, torch.float16, None, gen, rng)
    # (n_sqnorm or 0 for none, max_norm, grad_scale, weight decay, step); max_norm 1e6: coefficient >= 1
    cases = [(0, 1.0, 1.0, 0.0, 1), (1, 0.0, 1.0, 0.1, 1), (1, 1e6, 1.0, 0.1, 10000), (1, 1e-3, 1.0, 0.0, 2),
             (2, 0.5, 2.0, 0.1, 3), (255, 0.5, 0.5, 0.0, 10000), (256, 1e-2, 1.0, 0.1, 1), (257, 0.3, 0.25, 0.0, 7),
             (4097, 0.1, 3.0, 0.1, 10000), (4097, 1e6, 0.5, 0.0, 1)]
    for n_sq, max_norm, grad_scale, wd, step in cases:
        _run_adam_case(ops, 1032, torch.bfloat16, torch.float16, None, gen, rng, n_sq=n_sq, max_norm=max_norm,
                       grad_scale=grad_scale, wd=wd, step=step)


@pytest.mark.parametrize("clip", [False, True])
def test_compact_adam_non_finite_gradients(ops, clip):
    """A NaN and an Inf gradient element: the state at those positions follows IEEE arithmetic exactly as the oracle
    does.  With the clip, the norm (smt_grad_sqnorm) is NaN or Inf: a NaN coefficient is not < 1 (no clip), an Inf norm
    gives a zero coefficient (every finite gradient scaled to 0, Inf * 0 = NaN)."""
    gen = torch.Generator().manual_seed(2)
    rng = np.random.RandomState(2)
    n = 64 * 64 * 2
    blocks = [(0, 1), (1, 0)]
    cases = ([(100, float("nan")), (2000, float("inf"))], [(5000, float("inf"))], [(7, float("nan"))])
    for specials in cases:
        g = torch.from_numpy(rng.randn(n).astype(np.float32) * 0.05).bfloat16()
        for i, val in specials:
            g[i] = val
        if clip:
            sq = ops.grad_sqnorm(g.cuda())
            total = sq.item()
            p, m, v = _state(n, rng)
            gscale = _gscale(total, 0.5, 1.0)
            wp, wm, wv = _oracle_step(p, m, v, g.float().numpy(), 4, gscale, 0.01)
            dp, dm, dv = (torch.from_numpy(x.copy()).cuda() for x in (p, m, v))
            buf, W, (r0, c0) = _block_weight(2, 2, 64, torch.float16, gen)
            tab = ops.make_block_table([(W, r, c) for r, c in blocks], "cuda")
            comp = torch.empty(n, dtype=torch.bfloat16, device="cuda")
            ops.compact_adam(dp, dm, dv, g.cuda(), step=4, grad_scale=0.5, sqnorm=sq, max_norm=1.0, compact_out=comp,
                             weight_decay=0.01, table=tab, n_blocks=2, block=64, w_dtype=torch.float16, **HP)
            _np_same(dp.cpu().numpy(), wp, "master")
            _np_same(dm.cpu().numpy(), wm, "exp_avg")
            _np_same(dv.cpu().numpy(), wv, "exp_avg_sq")
            _same(comp, torch.from_numpy(wp).bfloat16(), "compact")
            got_w = torch.cat([W[r * 64:(r + 1) * 64, c * 64:(c + 1) * 64].reshape(-1) for r, c in blocks])
            _same(got_w, torch.from_numpy(wp).half(), "W")
            assert np.isnan(wp).any()
        else:
            _run_adam_case(ops, 0, torch.bfloat16, torch.float32, torch.bfloat16, gen, rng, blocks=blocks,
                           rbcb=(2, 2), n_sq=0, g=g, step=4)


@pytest.mark.parametrize("wdt", [torch.float32, torch.float16])
def test_compact_adam_columns_multi_pass(ops, sms, wdt):
    """More table entries than one pass of the grid (SMs x 8 CTAs x 8 entries), n_out = 8 and 136 (not a multiple of
    the 128-row tile), weights as views with ldw > in_features, gaps of uncovered arena elements."""
    gen = torch.Generator().manual_seed(wdt.itemsize)
    rng = np.random.RandomState(wdt.itemsize)
    need = sms * 8 * 8 + 37
    per_w = need // 2 + 1
    F = per_w + 40
    weights, bufs = [], []
    for out_f in (8, 136):
        buf = torch.full((out_f, F + 13), -0.375, dtype=wdt)
        buf[:, 3:3 + F] = torch.randn(out_f, F, generator=gen).to(wdt)
        buf = buf.cuda()
        bufs.append(buf)
        weights.append(buf[:, 3:3 + F])
    entries = [(w, c) for w in (0, 1) for c in torch.randperm(F, generator=gen)[:per_w].tolist()]
    entries = [entries[i] for i in torch.randperm(len(entries), generator=gen).tolist()]
    offs, off = [], 0
    for i, (w, _c) in enumerate(entries):
        if i % 5 == 0:
            off += 8                                              # uncovered arena elements
        offs.append(off)
        off += weights[w].shape[0]
    n = off + 16
    covered = np.zeros(n, bool)
    for (w, _c), o in zip(entries, offs):
        covered[o:o + weights[w].shape[0]] = True
    table = ops.make_column_table([(weights[w], c, o) for (w, c), o in zip(entries, offs)], "cuda")
    p, m, v = _state(n, rng)
    g = torch.from_numpy(rng.randn(n).astype(np.float32) * 0.05).bfloat16()
    parts = (rng.rand(7) * 0.02).astype(np.float32)
    gscale = _gscale(O.partial_sqnorm_total(parts), 0.5, 1.0)
    wp, wm, wv = _oracle_step(p, m, v, g.float().numpy(), 5, gscale, 0.01)
    kw = dict(step=5, grad_scale=0.5, sqnorm=torch.from_numpy(parts).cuda(), max_norm=1.0, weight_decay=0.01, **HP)
    # the block kernel over the whole arena: the column kernel must match it bit for bit on the covered elements
    bp, bm, bv = (torch.from_numpy(x.copy()).cuda() for x in (p, m, v))
    ops.compact_adam(bp, bm, bv, g.cuda(), **kw)
    before = [b.cpu() for b in bufs]
    runs = []
    for _ in range(2):
        for b, h in zip(bufs, before):
            b.copy_(h)
        dp, dm, dv = (torch.from_numpy(x.copy()).cuda() for x in (p, m, v))
        comp = torch.full((n,), -2.0, dtype=torch.float16, device="cuda")
        ops.compact_adam(dp, dm, dv, g.cuda(), compact_out=comp, columns=table, n_columns=len(entries),
                         w_dtype=wdt, **kw)
        for got, want, init, blk, what in ((dp, wp, p, bp, "master"), (dm, wm, m, bm, "exp_avg"),
                                          (dv, wv, v, bv, "exp_avg_sq")):
            got = got.cpu().numpy()
            _np_same(got[covered], want[covered], what)
            _np_same(got[covered], blk.cpu().numpy()[covered], what + " vs compact_adam")
            _np_same(got[~covered], init[~covered], what + " uncovered")
        cc = comp.cpu()
        _same(cc[torch.from_numpy(covered)], torch.from_numpy(wp[covered]).half(), "compact")
        assert (cc[torch.from_numpy(~covered)] == -2.0).all()
        master = torch.from_numpy(wp)
        for wi, buf in enumerate(bufs):
            expect = before[wi].clone()
            for (w, c), o in zip(entries, offs):
                if w == wi:
                    expect[:, 3 + c] = master[o:o + expect.shape[0]].to(wdt)
            _same(buf, expect, ("W", wi))
        runs.append([dp.cpu(), dm.cpu(), dv.cpu(), cc] + [b.cpu() for b in bufs])
    assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(*runs))
