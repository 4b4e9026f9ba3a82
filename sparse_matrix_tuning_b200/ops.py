"""Tensor-level wrappers over the C-ABI: one Python function per entry point of `include/smt_b200.h`.

PyTorch is used for device memory and streams only; all arithmetic happens in libsmt_b200.so.
Every function launches on the CURRENT CUDA stream of the tensors' device.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import BlockRef, check, dtype_id, load, ptr, require_cuda, stream_ptr

STRATEGY_IDS = _lib.STRATEGY_IDS

# ---- instrumentation (bench.py): number of OUR kernels launched, optional CUDA-event timing of one op -------
LAUNCHES = {"total": 0}
_timers: dict = {}


def _req(cond: bool, what: str) -> None:
    """Argument validation that survives `python -O` (unlike assert): the C-ABI trusts these shapes."""
    if not cond:
        raise _lib.SMTLibraryError(f"invalid argument: expected {what}")


def _count(n: int = 1) -> None:
    LAUNCHES["total"] += n


def enable_timing(op_name: str, enabled: bool = True) -> None:
    """Bracket every call of `op_name` ('block_grad_gemm', 'compact_adam', ...) with CUDA events recorded on the
    launching stream; read the durations with `collect_timing` after a synchronize."""
    if enabled:
        _timers[op_name] = []
    else:
        _timers.pop(op_name, None)


def collect_timing(op_name: str, reset: bool = True):
    """[(milliseconds, tag), ...] for the bracketed calls since the last reset (synchronizes the events)."""
    rec = _timers.get(op_name, [])
    out = [(a.elapsed_time(b), tag) for a, b, tag in rec]
    if reset and op_name in _timers:
        _timers[op_name] = []
    return out


class _timed:
    def __init__(self, op_name, device, tag=None):
        self.rec = _timers.get(op_name)
        self.device, self.tag = device, tag

    def __enter__(self):
        if self.rec is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record(torch.cuda.current_stream(self.device))
        return self

    def __exit__(self, *exc):
        if self.rec is not None:
            self.b.record(torch.cuda.current_stream(self.device))
            self.rec.append((self.a, self.b, self.tag))
        return False


def _st(t: torch.Tensor) -> int:
    return stream_ptr(t.device)


# ---- block tables --------------------------------------------------------------------------------

def make_block_table(entries: Sequence[Tuple[torch.Tensor, int, int]], device) -> torch.Tensor:
    """Device array of `smt_block_ref` for [(weight, block_row, block_col), ...] (uint8 tensor view)."""
    n = len(entries)
    arr = (BlockRef * max(n, 1))()
    for i, (w, r, c) in enumerate(entries):
        if w.dim() != 2 or w.stride(1) != 1:
            raise _lib.SMTLibraryError("block table: weights must be 2-D with unit column stride")
        if w.data_ptr() % 16 != 0 or (w.stride(0) * w.element_size()) % 16 != 0:
            # the copy / write-back kernels move 128-bit vectors; a weight re-pointed into a flat buffer at an odd
            # offset must be rejected here (the C entry points cannot see inside the device-resident table)
            raise _lib.SMTLibraryError("block table: weight storage must be 16-byte aligned (pointer and row pitch); "
                                       f"got data_ptr % 16 = {w.data_ptr() % 16}, row pitch = "
                                       f"{w.stride(0) * w.element_size()} B")
        arr[i].w_ptr = w.data_ptr()
        arr[i].ldw = w.stride(0)
        arr[i].row = int(r)
        arr[i].col = int(c)
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)[: n * C.sizeof(BlockRef)].clone()
    return host.to(device)


def make_block_rc(index_list: Sequence[Tuple[int, int]], device) -> torch.Tensor:
    """Device int32 [n, 2] table of (block_row, block_col) — the reference's `index_list`."""
    if len(index_list) == 0:
        return torch.empty((0, 2), dtype=torch.int32, device=device)
    return torch.tensor([[int(r), int(c)] for r, c in index_list], dtype=torch.int32, device=device)


# ---- warm-up scoring -------------------------------------------------------------------------------

def score_accumulate(acc: torch.Tensor, grad: torch.Tensor) -> None:
    """acc += grad (fp32 accumulator, any supported grad dtype). fine_tune.py:724-765."""
    require_cuda(acc, grad)
    _req(acc.dtype == torch.float32 and acc.is_contiguous() and grad.is_contiguous(),
         "acc.dtype == torch.float32 and acc.is_contiguous() and grad.is_contiguous()")
    _req(acc.numel() == grad.numel(), "acc.numel() == grad.numel()")
    check(load().smt_score_accumulate(ptr(acc), ptr(grad), dtype_id(grad.dtype), grad.numel(), _st(acc)),
          "smt_score_accumulate")
    _count()


def block_sum_accumulate(block_sums: torch.Tensor, grad: torch.Tensor, block: int) -> None:
    """block_sums[R/b, C/b] += per-block signed sums of grad[R, C]."""
    require_cuda(block_sums, grad)
    _req(grad.dim() == 2 and grad.stride(1) == 1 and block_sums.dtype == torch.float32,
         "grad.dim() == 2 and grad.stride(1) == 1 and block_sums.dtype == torch.float32")
    R, Cc = grad.shape
    _req(block_sums.is_contiguous() and block_sums.numel() == (R // block) * (Cc // block),
         "block_sums.is_contiguous() and block_sums.numel() == (R // block) * (Cc // block)")
    check(load().smt_block_sum_accumulate(ptr(block_sums), ptr(grad), dtype_id(grad.dtype), R, Cc,
                                          grad.stride(0), block, _st(grad)), "smt_block_sum_accumulate")
    _count()


def block_sum_finalize(block_sums: torch.Tensor, block: int) -> torch.Tensor:
    require_cuda(block_sums)
    out = torch.empty_like(block_sums)
    check(load().smt_block_sum_finalize(ptr(block_sums), ptr(out), block_sums.numel(), block, _st(out)),
          "smt_block_sum_finalize")
    _count()
    return out


def block_score_reduce(acc: torch.Tensor, block: int, strategy: str = "mean_abs",
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """scores[R/b, C/b] of an fp32 [R, C] matrix. smt_helper.py:55-78, 233-251."""
    require_cuda(acc)
    _req(acc.dim() == 2 and acc.dtype == torch.float32 and acc.stride(1) == 1,
         "acc.dim() == 2 and acc.dtype == torch.float32 and acc.stride(1) == 1")
    if strategy not in STRATEGY_IDS:
        raise _lib.SMTLibraryError(f"unknown calculate_strategy {strategy!r}")
    R, Cc = acc.shape
    if out is None:
        out = torch.empty((R // block, Cc // block), dtype=torch.float32, device=acc.device)
    check(load().smt_block_score_reduce(ptr(acc), R, Cc, acc.stride(0), block, STRATEGY_IDS[strategy],
                                        ptr(out), _st(acc)), "smt_block_score_reduce")
    _count()
    return out


def token_block_sums(t2d: torch.Tensor, block: int) -> torch.Tensor:
    """out[t, j] = sum_{k < b} t2d[t, j*b + k] as fp32 [T, F/b]: the per-token block sums of a module's input or output
    gradient that `block_outer_accumulate` contracts into weight-gradient block sums (fine_tune.py:716-768 and
    smt_helper.py:55-78 without the weight gradient)."""
    require_cuda(t2d)
    _req(t2d.dim() == 2 and t2d.stride(1) == 1, "t2d.dim() == 2 and t2d.stride(1) == 1")
    T, F = t2d.shape
    _req(block in (64, 128, 256) and F % block == 0, "block in (64, 128, 256) and F % block == 0")
    out = torch.empty((T, F // block), dtype=torch.float32, device=t2d.device)
    check(load().smt_token_block_sums(ptr(t2d), dtype_id(t2d.dtype), T, F, t2d.stride(0) if T > 0 else F, block,
                                      ptr(out), _st(t2d)), "smt_token_block_sums")
    if T > 0 and F > 0:
        _count()
    return out


def block_outer_accumulate(block_sums: torch.Tensor, dy_sums: torch.Tensor, x_sums: torch.Tensor) -> None:
    """block_sums[r, c] += sum_t dy_sums[t, r] * x_sums[t, c] (fp32, deterministic: a fixed partition of T)."""
    require_cuda(block_sums, dy_sums, x_sums)
    for t in (block_sums, dy_sums, x_sums):
        _req(t.dim() == 2 and t.dtype == torch.float32 and t.is_contiguous(), "contiguous 2-D fp32 tensors")
    T, rb = dy_sums.shape
    cb = x_sums.shape[1]
    _req(x_sums.shape[0] == T and tuple(block_sums.shape) == (rb, cb),
         "dy_sums [T, rb], x_sums [T, cb] and block_sums [rb, cb]")
    lib = load()
    ws_bytes = lib.smt_block_outer_accumulate_workspace_bytes(T, rb, cb)
    ws = _workspace(ws_bytes, block_sums.device, tag="block_outer")
    check(lib.smt_block_outer_accumulate(ptr(block_sums), ptr(dy_sums), ptr(x_sums), T, rb, cb, ptr(ws), ws_bytes,
                                         _st(block_sums)), "smt_block_outer_accumulate")
    if T > 0 and rb * cb > 0:
        _count(2)


def act_score_accumulate(acc: torch.Tensor, x: torch.Tensor) -> None:
    """acc[S, C] += sum_b |x[b, S, C]|. fine_tune.py:649-678 (reduced over batch)."""
    require_cuda(acc, x)
    _req(x.dim() == 3 and x.is_contiguous() and acc.is_contiguous() and acc.dtype == torch.float32,
         "x.dim() == 3 and x.is_contiguous() and acc.is_contiguous() and acc.dtype == torch.float32")
    Bn, S, Cc = x.shape
    _req(tuple(acc.shape) == (S, Cc), "tuple(acc.shape) == (S, Cc)")
    check(load().smt_act_score_accumulate(ptr(acc), ptr(x), dtype_id(x.dtype), Bn, S, Cc, _st(x)),
          "smt_act_score_accumulate")
    _count()


def channel_score_reduce(acc: torch.Tensor, strategy: str = "mean_abs") -> torch.Tensor:
    require_cuda(acc)
    _req(acc.dim() == 2 and acc.is_contiguous() and acc.dtype == torch.float32,
         "acc.dim() == 2 and acc.is_contiguous() and acc.dtype == torch.float32")
    if strategy not in STRATEGY_IDS:
        raise _lib.SMTLibraryError(f"unknown calculate_strategy {strategy!r}")
    S, Cc = acc.shape
    out = torch.empty((Cc,), dtype=torch.float32, device=acc.device)
    check(load().smt_channel_score_reduce(ptr(acc), S, Cc, STRATEGY_IDS[strategy], ptr(out), _st(acc)),
          "smt_channel_score_reduce")
    _count()
    return out


# ---- top-k -----------------------------------------------------------------------------------------

def topk_blocks(scores: torch.Tensor, seg_offsets: Sequence[int], seg_k: Sequence[int],
                tiebreak_rank: Optional[torch.Tensor] = None,
                inv_rank: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, list]:
    """Segmented top-k. Returns (flat int32 indices on device, per-segment output offsets (host list))."""
    require_cuda(scores, tiebreak_rank, inv_rank)
    _req(scores.dtype == torch.float32 and scores.is_contiguous(),
         "scores.dtype == torch.float32 and scores.is_contiguous()")
    n = scores.numel()
    nseg = len(seg_k)
    _req(len(seg_offsets) == nseg + 1 and seg_offsets[-1] == n,
         "len(seg_offsets) == nseg + 1 and seg_offsets[-1] == n")
    out_offsets = [0]
    for s in range(nseg):
        length = seg_offsets[s + 1] - seg_offsets[s]
        out_offsets.append(out_offsets[-1] + max(0, min(int(seg_k[s]), length)))
    dev = scores.device
    d_off = torch.tensor(list(seg_offsets), dtype=torch.int32, device=dev)
    d_k = torch.tensor([int(k) for k in seg_k], dtype=torch.int32, device=dev)
    d_out_off = torch.tensor(out_offsets, dtype=torch.int32, device=dev)
    out = torch.empty((max(out_offsets[-1], 1),), dtype=torch.int32, device=dev)
    lib = load()
    ws_bytes = lib.smt_topk_workspace_bytes(n)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    if tiebreak_rank is not None:
        _req(tiebreak_rank.dtype == torch.int32 or tiebreak_rank.dtype == torch.uint32,
             "tiebreak_rank.dtype == torch.int32 or tiebreak_rank.dtype == torch.uint32")
        _req(inv_rank is not None and inv_rank.numel() == n and tiebreak_rank.numel() == n,
             "inv_rank is not None and inv_rank.numel() == n and tiebreak_rank.numel() == n")
    check(lib.smt_topk_blocks(ptr(scores), ptr(tiebreak_rank), ptr(inv_rank), n, ptr(d_off), ptr(d_k),
                              ptr(d_out_off), nseg, ptr(out), ptr(ws), ws_bytes, _st(scores)),
          "smt_topk_blocks")
    _count()
    return out[: out_offsets[-1]], out_offsets


# ---- gather / scatter ---------------------------------------------------------------------------------

def block_gather(table: torch.Tensor, n_blocks: int, block: int, compact: torch.Tensor) -> None:
    """compact[i] <- W_i block. smt.py:317-325."""
    require_cuda(table, compact)
    _req(compact.is_contiguous() and compact.numel() == n_blocks * block * block,
         "compact.is_contiguous() and compact.numel() == n_blocks * block * block")
    check(load().smt_block_gather(ptr(table), n_blocks, block, compact.element_size(), ptr(compact),
                                  _st(compact)), "smt_block_gather")
    _count()


def block_scatter(table: torch.Tensor, n_blocks: int, block: int, compact: torch.Tensor) -> None:
    """W_i block <- compact[i]. smt.py:332-341."""
    require_cuda(table, compact)
    _req(compact.is_contiguous() and compact.numel() == n_blocks * block * block,
         "compact.is_contiguous() and compact.numel() == n_blocks * block * block")
    check(load().smt_block_scatter(ptr(table), n_blocks, block, compact.element_size(), ptr(compact),
                                   _st(compact)), "smt_block_scatter")
    _count()


# ---- channel (input-column) movement ------------------------------------------------------------------------

def make_channel_idx(index_list, device, pad_to: int = 1) -> torch.Tensor:
    """int32 device copy of a channel index list, optionally padded with -1 ("no channel": channel_gather writes a zero
    column there) to a multiple of `pad_to`."""
    idx = [int(i) for i in index_list]
    idx += [-1] * (-len(idx) % pad_to)
    return torch.tensor(idx, dtype=torch.int32, device="cpu").to(device)


def channel_gather(x2: torch.Tensor, idx: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[t, i] = x2[t, idx[i]] — the packed selected input channels (smt.py:240-247)."""
    require_cuda(x2, idx)
    _req(x2.dim() == 2 and x2.stride(1) == 1 and idx.dtype == torch.int32 and idx.is_contiguous(),
         "x2.dim() == 2 and x2.stride(1) == 1 and idx.dtype == torch.int32 and idx.is_contiguous()")
    T, n = x2.shape[0], idx.numel()
    if out is None:
        out = torch.empty(T, n, dtype=x2.dtype, device=x2.device)
    _req(out.is_contiguous() and out.shape == (T, n) and out.dtype == x2.dtype,
         "out.is_contiguous() and out.shape == (T, n) and out.dtype == x2.dtype")
    check(load().smt_channel_gather(ptr(x2), T, x2.stride(0), ptr(idx), n, x2.element_size(), ptr(out), _st(x2)),
          "smt_channel_gather")
    _count()
    return out


def _column_args(W, idx, compact):
    require_cuda(W, idx, compact)
    _req(W.dim() == 2 and W.stride(1) == 1 and idx.dtype == torch.int32 and idx.is_contiguous(),
         "W.dim() == 2 and W.stride(1) == 1 and idx.dtype == torch.int32 and idx.is_contiguous()")
    n = idx.numel()
    _req(compact.is_contiguous() and compact.shape == (n, W.shape[0]) and compact.dtype == W.dtype,
         "compact.is_contiguous() and compact.shape == (n, W.shape[0]) and compact.dtype == W.dtype")
    return ptr(W), W.stride(0), W.shape[0], W.shape[1], ptr(idx), n, W.element_size(), ptr(compact), _st(W)


def column_gather(W: torch.Tensor, idx: torch.Tensor, compact: torch.Tensor) -> None:
    """compact[i, :] <- W[:, idx[i]]."""
    check(load().smt_column_gather(*_column_args(W, idx, compact)), "smt_column_gather")
    _count()


def column_scatter(W: torch.Tensor, idx: torch.Tensor, compact: torch.Tensor) -> None:
    """W[:, idx[i]] <- compact[i, :]."""
    check(load().smt_column_scatter(*_column_args(W, idx, compact)), "smt_column_scatter")
    _count()


# ---- block-gradient GEMM --------------------------------------------------------------------------------

_ws_cache: dict = {}
_channel_items: dict = {}


def channel_grad_gemm(partial: torch.Tensor, n: int, dy2d: torch.Tensor) -> torch.Tensor:
    """grad[i, o] = sum_t partial[t, i] * dy[t, o] for the n selected input channels - the weight gradient of
    linearChannel.backward (smt.py:283-284: `partial_input^T @ grad_output`, summed over the batch) on the tcgen05
    block-gradient pipeline: the packed channels play the `dy` operand (their row blocks are padded by TMA zero fill),
    grad_output the `x` operand, and every (row block, column block) tile is stored with the row pitch of the result, so
    the tiles assemble the row-major [n, out_features] gradient directly.  fp32 accumulation over all tokens, ONE
    rounding.  `partial`: [T, n8] (n8 >= n, row pitch a multiple of 16 bytes, columns >= n zero); returns [n, out]."""
    require_cuda(partial, dy2d)
    _req(partial.dim() == 2 and dy2d.dim() == 2 and partial.shape[0] == dy2d.shape[0] and partial.dtype == dy2d.dtype,
         "partial.dim() == 2 and dy2d.dim() == 2 and partial.shape[0] == dy2d.shape[0] and partial.dtype == dy2d.dtype")
    _req(partial.stride(1) == 1 and dy2d.stride(1) == 1 and partial.dtype in (torch.bfloat16, torch.float16),
         "partial.stride(1) == 1 and dy2d.stride(1) == 1 and partial.dtype in (torch.bfloat16, torch.float16)")
    T, out_f = dy2d.shape
    _req(0 < n <= partial.shape[1] and (partial.stride(0) * 2) % 16 == 0 and (dy2d.stride(0) * 2) % 16 == 0,
         "0 < n <= partial.shape[1] and 16-byte row pitches")
    _req(out_f % 64 == 0, "out_features % 64 == 0")
    block = 128 if (out_f % 128 == 0 and n > 64) else 64
    rows, cols = (n + block - 1) // block, out_f // block
    dev = dy2d.device
    out = torch.empty(rows * block, out_f, dtype=dy2d.dtype, device=dev)
    if T == 0:
        return out.zero_()[:n]
    import numpy as np
    key = (rows, cols, block, out_f)
    arr = _channel_items.get(key)
    if arr is None:
        arr = np.array([(0, 1, r, c, r * block * out_f + c * block, _lib.ITEM_OVERWRITE, -1)
                        for r in range(rows) for c in range(cols)], dtype=_item_dtype())
        if len(_channel_items) > 64:
            _channel_items.clear()
        _channel_items[key] = arr
    lib = load()
    n_items = len(arr)
    stage = torch.empty(2 * 128 + arr.nbytes, dtype=torch.uint8, pin_memory=True)
    in_id = dtype_id(dy2d.dtype)
    check(lib.smt_encode_operand_map(stage.data_ptr(), partial.data_ptr(), partial.shape[1], T, partial.stride(0),
                                     in_id, block), "smt_encode_operand_map")
    check(lib.smt_encode_operand_map(stage.data_ptr() + 128, dy2d.data_ptr(), out_f, T, dy2d.stride(0), in_id, block),
          "smt_encode_operand_map")
    stage.numpy()[256:] = arr.view("u1").reshape(-1)
    dev_buf = stage.to(dev, non_blocking=True)
    ws_bytes = lib.smt_block_grad_gemm_grouped_workspace_bytes(n_items, block, T)
    ws = _workspace(ws_bytes, dev)
    with _timed("channel_grad_gemm", dev, (n, out_f, T)):
        check(lib.smt_block_grad_gemm_grouped(dev_buf.data_ptr(), dev_buf.data_ptr() + 256, n_items, T, block, in_id,
                                              out.data_ptr(), dtype_id(out.dtype), 0, out_f, 0, ptr(ws), ws_bytes,
                                              stream_ptr(dev)), "smt_block_grad_gemm_grouped")
    _count(lib.smt_last_launch_count())
    return out[:n]


def _workspace(nbytes: int, device, tag: str = "gemm") -> Optional[torch.Tensor]:
    """Grow-only per-(purpose, device, stream) scratch buffer (allocation stays out of the C library).  Buffers are
    ZERO-initialised when (re)allocated: the GEMM keeps self-resetting split-K arrival counters in the first 16 KiB
    of its workspace (see smt_block_grad_gemm in include/smt_b200.h)."""
    if nbytes == 0:
        return None
    key = (tag, device, torch.cuda.current_stream(device).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.zeros((nbytes,), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


_runs_cache: dict = {}
LAST_SINGLE: dict = {}    # which kernel the last single-problem block_grad_gemm used (tests / reports)


def _runs_for(index_list, block: int, device):
    """Strip-sharing runs of an index list (cached per list object, validated by value): blocks grouped by block row,
    columns ascending, cut into runs of at most `run width` blocks; b = 256 yields one run per 128-row half.
    Returns (device tensor of smt_gemm_run, number of runs, fraction of the blocks that sit in a run of >= 2)."""
    import numpy as np
    snap = _snapshot_index_list(index_list)
    key = (id(index_list), block, device)
    hit = _runs_cache.get(key)
    if hit is not None and hit[0] is snap:
        return hit[1]
    width = load().smt_block_grad_gemm_run_width(block)
    by_row: dict = {}
    for i, (r, c) in enumerate(snap):
        by_row.setdefault(r, []).append((c, i))
    rows, shared = [], 0
    for r in sorted(by_row):
        cols = sorted(by_row[r])
        for k in range(0, len(cols), width):
            part = cols[k:k + width]
            if len(part) >= 2:
                shared += len(part)
            for half in ((0, 1) if block == 256 else (0,)):
                cs = [c for c, _ in part] + [0] * (4 - len(part))
                bs = [i for _, i in part] + [0] * (4 - len(part))
                rows.append((r, half, len(part), *cs, *bs, 0))
    arr = np.array(rows, dtype=np.int32).reshape(-1, 12)
    assert arr.shape[1] * 4 == C.sizeof(_lib.GemmRun)
    dev = torch.from_numpy(arr).to(device) if len(rows) else torch.empty((0, 12), dtype=torch.int32, device=device)
    res = (dev, len(rows), shared / max(len(snap), 1))
    if len(_runs_cache) > 4096:
        _runs_cache.clear()
    _runs_cache[key] = (snap, res)
    return res


def block_grad_gemm(x2d: torch.Tensor, dy2d: torch.Tensor, block_rc: torch.Tensor, block: int,
                    out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
                    accumulate: bool = False, index_list=None) -> torch.Tensor:
    """G[i*b+o, k] (+)= sum_t dy[t, r_i*b+o] * x[t, c_i*b+k]. smt.py:386-404.

    x2d: [T, in], dy2d: [T, out] (unit column stride, same dtype); block_rc: int32 [n, 2] on device.
    `index_list` (optional): the host-side list `block_rc` was made from.  With it, 16-bit launches in which enough
    blocks share a block row run the strip-sharing kernel (`smt_block_grad_gemm_runs`: the dy strip is fetched once per
    run of up to 4 / 2 / 2 blocks for b = 64 / 128 / 256).  SMT_GEMM_RUNS=0 disables that, =2 forces it.
    """
    require_cuda(x2d, dy2d, block_rc)
    _req(x2d.dim() == 2 and dy2d.dim() == 2 and x2d.shape[0] == dy2d.shape[0],
         "x2d.dim() == 2 and dy2d.dim() == 2 and x2d.shape[0] == dy2d.shape[0]")
    _req(x2d.stride(1) == 1 and dy2d.stride(1) == 1 and x2d.dtype == dy2d.dtype,
         "x2d.stride(1) == 1 and dy2d.stride(1) == 1 and x2d.dtype == dy2d.dtype")
    _req(block_rc.dtype == torch.int32 and block_rc.is_contiguous(),
         "block_rc.dtype == torch.int32 and block_rc.is_contiguous()")
    n = block_rc.shape[0]
    T = x2d.shape[0]
    if out is None:
        out = torch.empty((n * block, block), dtype=out_dtype or dy2d.dtype, device=x2d.device)
        accumulate = False
    _req(out.is_contiguous() and out.numel() == n * block * block,
         "out.is_contiguous() and out.numel() == n * block * block")
    lib = load()
    in_id = dtype_id(x2d.dtype)
    import os
    mode = os.environ.get("SMT_GEMM_RUNS", "1")
    if index_list is not None and mode != "0" and n > 0 and T > 0 and x2d.dtype != torch.float32:
        _req(len(index_list) == n, "len(index_list) == block_rc.shape[0]")
        runs, n_runs, shared = _runs_for(index_list, block, x2d.device)
        # Measured rule (profiles/r02_kernel_sweep.md): run tiles pay when the launch is big enough for the operand feed
        # to matter (>= 148 blocks), the runs are wide (singles are better off on the plain kernel's taller stages;
        # two 80 KiB stages of a b = 256 pair tile cannot hide HBM latency) and the run tiles (times their one-wave
        # split factor) still fill the GPU.  Small launches are bound by fixed costs either way.
        width = n / max(n_runs, 1)
        sms = 148
        fill = n_runs if n_runs >= sms else n_runs * (sms // max(n_runs, 1))      # CTAs of the (one-wave) split plan
        if mode == "2" or (block != 256 and n >= 148 and width >= (2.0 if block == 64 else 1.5) and fill >= 80):
            ws_bytes = lib.smt_block_grad_gemm_runs_workspace_bytes(n_runs, block, T)
            ws = _workspace(ws_bytes, x2d.device, tag="gemm_runs")
            with _timed("block_grad_gemm", x2d.device, (n, block, T)):
                check(lib.smt_block_grad_gemm_runs(ptr(x2d), x2d.stride(0), x2d.shape[1], ptr(dy2d), dy2d.stride(0),
                                                   dy2d.shape[1], T, in_id, ptr(runs), n_runs, block, ptr(out),
                                                   dtype_id(out.dtype), 1 if accumulate else 0, ptr(ws), ws_bytes,
                                                   _st(x2d)), "smt_block_grad_gemm_runs")
            _count(lib.smt_last_launch_count())
            LAST_SINGLE.update(kernel="runs", runs=n_runs, shared_fraction=shared)
            return out
    LAST_SINGLE.update(kernel="blocks", runs=0, shared_fraction=0.0)
    ws_bytes = lib.smt_block_grad_gemm_workspace_bytes(n, block, T, in_id)
    ws = _workspace(ws_bytes, x2d.device)
    with _timed("block_grad_gemm", x2d.device, (n, block, T)):
        check(lib.smt_block_grad_gemm(ptr(x2d), x2d.stride(0) if T > 0 else x2d.shape[1], x2d.shape[1],
                                      ptr(dy2d), dy2d.stride(0) if T > 0 else dy2d.shape[1], dy2d.shape[1],
                                      T, in_id, ptr(block_rc), n, block, ptr(out), dtype_id(out.dtype),
                                      1 if accumulate else 0, ptr(ws), ws_bytes, _st(x2d)),
              "smt_block_grad_gemm")
    if n > 0 and T > 0:
        _count(lib.smt_last_launch_count())
    return out


def block_grad_gemm_plan(n_blocks: int, block: int, T: int, dtype: torch.dtype) -> Tuple[int, int]:
    a, b = C.c_int(), C.c_int()
    check(load().smt_block_grad_gemm_plan(n_blocks, block, T, dtype_id(dtype), C.byref(a), C.byref(b)),
          "smt_block_grad_gemm_plan")
    return a.value, b.value


# ---- dense side of linearZ, fused over modules that share their input ---------------------------------------------

def fused_linear_supported(weights: Sequence[torch.Tensor], dgrad: bool = False) -> bool:
    """True when `fused_linear_forward` / `fused_linear_dgrad` can take these weights (1-3 [N_j, K] matrices of one
    16-bit dtype on one CUDA device with aligned storage); the caller keeps the per-module library GEMMs otherwise."""
    if not 1 <= len(weights) <= 3:
        return False
    w0 = weights[0]
    if not w0.is_cuda or w0.dtype not in (torch.bfloat16, torch.float16):
        return False
    for w in weights:
        if w.dim() != 2 or w.dtype != w0.dtype or w.device != w0.device or w.shape[1] != w0.shape[1] or w.stride(1) != 1:
            return False
        if w.data_ptr() % 16 or (w.stride(0) * 2) % 16:
            return False
    ns = (C.c_int * len(weights))(*[int(w.shape[0]) for w in weights])
    return bool(load().smt_fused_linear_supported(len(weights), ns, int(w0.shape[1]), dtype_id(w0.dtype), 1 if dgrad else 0))


def _seg_arrays(tensors: Sequence[torch.Tensor]):
    n = len(tensors)
    ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
    lds = (C.c_int64 * n)(*[t.stride(0) for t in tensors])
    return ptrs, lds


def fused_linear_forward(x2d: torch.Tensor, weights: Sequence[torch.Tensor]) -> list:
    """[x2d @ W_j^T for j] in ONE tcgen05 launch (smt.py:366 for every module that reads x).  x2d: [T, K]."""
    require_cuda(x2d, *weights)
    _req(x2d.dim() == 2 and x2d.stride(1) == 1 and x2d.dtype == weights[0].dtype and x2d.shape[1] == weights[0].shape[1],
         "x2d.dim() == 2 and x2d.stride(1) == 1 and x2d.dtype == weights[0].dtype and x2d.shape[1] == K")
    _req(x2d.data_ptr() % 16 == 0 and (x2d.stride(0) * 2) % 16 == 0, "16-byte aligned x")
    T, K = x2d.shape
    ys = [torch.empty(T, w.shape[0], dtype=x2d.dtype, device=x2d.device) for w in weights]
    n = len(weights)
    wp, wl = _seg_arrays(weights)
    yp, yl = _seg_arrays(ys)
    ns = (C.c_int * n)(*[int(w.shape[0]) for w in weights])
    with _timed("fused_linear_forward", x2d.device, (T, K, sum(w.shape[0] for w in weights))):
        check(load().smt_fused_linear_forward(ptr(x2d), x2d.stride(0) if T > 0 else K, T, K, n, wp, wl, ns, yp, yl,
                                              dtype_id(x2d.dtype), _st(x2d)), "smt_fused_linear_forward")
    if T > 0:
        _count()
    return ys


def fused_linear_dgrad(dys: Sequence[torch.Tensor], weights: Sequence[torch.Tensor],
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """sum_j dy_j @ W_j in ONE tcgen05 launch (smt.py:406 for every module that reads x, plus autograd's adds).
    `out`: optional [T, K] destination with unit column stride (e.g. a row slice of a larger buffer)."""
    require_cuda(*dys, *weights)
    _req(len(dys) == len(weights) and len(dys) >= 1, "len(dys) == len(weights) >= 1")
    T, K = dys[0].shape[0], weights[0].shape[1]
    for dy, w in zip(dys, weights):
        _req(dy.dim() == 2 and dy.stride(1) == 1 and dy.shape == (T, w.shape[0]) and dy.dtype == w.dtype,
             "dy.dim() == 2 and dy.stride(1) == 1 and dy.shape == (T, N_j) and dy.dtype == w.dtype")
        _req(dy.data_ptr() % 16 == 0 and (dy.stride(0) * 2) % 16 == 0, "16-byte aligned dy")
    if out is None:
        dx = torch.empty(T, K, dtype=dys[0].dtype, device=dys[0].device)
    else:
        require_cuda(out)
        _req(out.shape == (T, K) and out.dtype == dys[0].dtype and out.stride(1) == 1 and out.data_ptr() % 16 == 0
             and (out.stride(0) * 2) % 16 == 0, "out [T, K] of dy's dtype, unit column stride, 16-byte aligned rows")
        dx = out
    n = len(weights)
    wp, wl = _seg_arrays(weights)
    dp_, dl = _seg_arrays(dys)
    ns = (C.c_int * n)(*[int(w.shape[0]) for w in weights])
    with _timed("fused_linear_dgrad", dx.device, (T, K, sum(w.shape[0] for w in weights))):
        check(load().smt_fused_linear_dgrad(dp_, dl, T, K, n, wp, wl, ns, ptr(dx), dx.stride(0) if T > 0 else K,
                                            dtype_id(dx.dtype), _st(dx)), "smt_fused_linear_dgrad")
    if T > 0:
        _count()
    return dx


# ---- elementwise work of a LLaMA decoder layer (RMSNorm, RoPE, SwiGLU) ----------------------------------------------

def _bf16_operands(*ts) -> None:
    require_cuda(*ts)
    for t in ts:
        if t is not None:
            _req(t.dtype == torch.bfloat16 and t.is_contiguous() and t.data_ptr() % 16 == 0,
                 "contiguous, 16-byte aligned bfloat16 tensors")


def rmsnorm_forward(a: torch.Tensor, weight: torch.Tensor, eps: float, res: Optional[torch.Tensor] = None):
    """RMSNorm over the last dimension of `a` (or of h = bf16(res + a)).  Returns (y, rstd [rows] fp32, h or None)."""
    _bf16_operands(a, weight, res)
    H = a.shape[-1]
    _req(weight.shape == (H,) and (res is None or res.shape == a.shape), "weight [H] and res of a's shape")
    T = a.numel() // H if H else 0
    y = torch.empty_like(a)
    h = torch.empty_like(a) if res is not None else None
    rstd = torch.empty(T, dtype=torch.float32, device=a.device)
    check(load().smt_rmsnorm_forward(ptr(a), ptr(res), ptr(weight), T, H, float(eps), ptr(h), ptr(y), ptr(rstd), _st(a)),
          "smt_rmsnorm_forward")
    if T > 0:
        _count()
    return y, rstd, h


def rmsnorm_backward(x: torch.Tensor, weight: torch.Tensor, rstd: torch.Tensor, dy: torch.Tensor,
                     dres: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Input gradient of `rmsnorm_forward` for a frozen weight, plus `dres` (the residual stream's gradient) if given."""
    _bf16_operands(x, weight, dy, dres)
    H = x.shape[-1]
    T = x.numel() // H if H else 0
    _req(dy.shape == x.shape and (dres is None or dres.shape == x.shape) and weight.shape == (H,),
         "dy and dres of x's shape, weight [H]")
    _req(rstd.dtype == torch.float32 and rstd.is_contiguous() and rstd.numel() == T, "fp32 rstd with one entry per row")
    dx = torch.empty_like(x)
    check(load().smt_rmsnorm_backward(ptr(x), ptr(weight), ptr(rstd), ptr(dy), ptr(dres), T, H, ptr(dx), _st(x)),
          "smt_rmsnorm_backward")
    if T > 0:
        _count()
    return dx


def _rope(fn_name: str, q: torch.Tensor, k: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor):
    _bf16_operands(q, k)
    require_cuda(cos, sin)
    _req(q.dim() == 4 and k.dim() == 4 and q.shape[:2] == k.shape[:2] and q.shape[3] == 128 and k.shape[3] == 128,
         "q [B, S, Hq, 128] and k [B, S, Hk, 128]")
    B, S, Hq, _ = q.shape
    Hk = k.shape[2]
    _req(cos.shape == sin.shape and cos.dim() == 3 and cos.shape[1:] == (S, 128) and cos.shape[0] in (1, B)
         and cos.dtype == torch.bfloat16 and sin.dtype == torch.bfloat16, "bf16 cos / sin of shape [1 or B, S, 128]")
    _req(cos.stride() == sin.stride() and cos.stride()[1:] == (128, 1) and cos.data_ptr() % 16 == 0
         and sin.data_ptr() % 16 == 0 and cos.stride(0) % 8 == 0, "cos / sin with rows of 128 contiguous elements")
    bstride = 0 if cos.shape[0] == 1 else cos.stride(0)
    qo, ko = torch.empty_like(q), torch.empty_like(k)
    check(getattr(load(), fn_name)(ptr(q), ptr(k), ptr(cos), ptr(sin), B, S, Hq, Hk, bstride, ptr(qo), ptr(ko), _st(q)),
          fn_name)
    if q.numel() + k.numel() > 0:
        _count()
    return qo, ko


def rope_forward(q: torch.Tensor, k: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor):
    """HF `apply_rotary_pos_emb` on q [B, S, Hq, 128] and k [B, S, Hk, 128] (contiguous) in ONE launch."""
    return _rope("smt_rope_forward", q, k, cos, sin)


def rope_backward(dq_out: torch.Tensor, dk_out: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor):
    """Gradients of q and k through `rope_forward`, in ONE launch."""
    return _rope("smt_rope_backward", dq_out, dk_out, cos, sin)


def swiglu_forward(g: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """bf16(bf16(silu(g)) * u), elementwise."""
    _bf16_operands(g, u)
    _req(g.shape == u.shape and g.numel() % 8 == 0, "g and u of one shape, numel % 8 == 0")
    h = torch.empty_like(g)
    check(load().smt_swiglu_forward(ptr(g), ptr(u), g.numel(), ptr(h), _st(g)), "smt_swiglu_forward")
    if g.numel():
        _count()
    return h


def swiglu_backward(g: torch.Tensor, u: torch.Tensor, dh: torch.Tensor):
    """(dg, du) of `swiglu_forward` in ONE pass over g, u and dh."""
    _bf16_operands(g, u, dh)
    _req(g.shape == u.shape == dh.shape and g.numel() % 8 == 0, "g, u and dh of one shape, numel % 8 == 0")
    dg, du = torch.empty_like(g), torch.empty_like(u)
    check(load().smt_swiglu_backward(ptr(g), ptr(u), ptr(dh), g.numel(), ptr(dg), ptr(du), _st(g)),
          "smt_swiglu_backward")
    if g.numel():
        _count()
    return dg, du


# ---- causal-LM loss --------------------------------------------------------------------------------------------------

def cross_entropy_rows(logits: torch.Tensor, labels: torch.Tensor, scale: torch.Tensor,
                       ignore_index: int = -100) -> torch.Tensor:
    """Per-row cross-entropy of bf16 `logits` [T, V] against int64 `labels` [T]; returns the fp32 losses [T] (0 for
    `ignore_index`, NaN for a label outside [0, V)) and OVERWRITES `logits` with the gradient of sum(loss) * scale.
    `scale`: fp32 device scalar, read on the device."""
    require_cuda(logits, labels, scale)
    _req(logits.dim() == 2 and logits.dtype == torch.bfloat16 and logits.stride(1) == 1
         and logits.stride(0) % 8 == 0 and logits.data_ptr() % 16 == 0 and logits.shape[1] % 8 == 0,
         "bf16 logits [T, V] with V % 8 == 0, unit column stride, row pitch % 8 == 0 and 16-byte alignment")
    T, V = logits.shape
    _req(labels.dtype == torch.int64 and labels.is_contiguous() and labels.shape == (T,), "contiguous int64 labels [T]")
    _req(scale.dtype == torch.float32 and scale.numel() == 1, "fp32 scale with one element")
    loss = torch.empty(T, dtype=torch.float32, device=logits.device)
    check(load().smt_cross_entropy_rows(ptr(logits), logits.stride(0) if T > 0 else V, T, V, ptr(labels),
                                        int(ignore_index), ptr(scale), ptr(loss), _st(logits)),
          "smt_cross_entropy_rows")
    if T > 0:
        _count()
    return loss


# ---- optimizer ---------------------------------------------------------------------------------------------

def grad_sqnorm(grad: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Deterministic sum of squares of a flat gradient buffer -> fp32 scalar tensor on device."""
    require_cuda(grad)
    _req(grad.is_contiguous(), "grad.is_contiguous()")
    if out is None:
        out = torch.empty((1,), dtype=torch.float32, device=grad.device)
    lib = load()
    ws_bytes = lib.smt_grad_sqnorm_workspace_bytes()
    ws = _workspace(ws_bytes, grad.device, tag="sqnorm")
    check(lib.smt_grad_sqnorm(ptr(grad), dtype_id(grad.dtype), grad.numel(), ptr(out), ptr(ws), ws_bytes,
                              _st(grad)), "smt_grad_sqnorm")
    _count(2)
    return out


def compact_adam(master: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, grad: torch.Tensor,
                 *, lr: float, beta1: float, beta2: float, eps: float, weight_decay: float, step: int,
                 grad_scale: float = 1.0, sqnorm: Optional[torch.Tensor] = None, max_norm: float = 0.0,
                 compact_out: Optional[torch.Tensor] = None, table: Optional[torch.Tensor] = None,
                 n_blocks: int = 0, block: int = 0, w_dtype: Optional[torch.dtype] = None) -> None:
    """One fused AdamW step over flat compact state (+ clip, + dense write-back). See smt_b200.h."""
    require_cuda(master, exp_avg, exp_avg_sq, grad, sqnorm, compact_out, table)
    for t in (master, exp_avg, exp_avg_sq):
        _req(t.dtype == torch.float32 and t.is_contiguous() and t.numel() == grad.numel(),
             "t.dtype == torch.float32 and t.is_contiguous() and t.numel() == grad.numel()")
    _req(grad.is_contiguous(), "grad.is_contiguous()")
    n_sq = 0
    if sqnorm is not None:
        # one scalar (smt_grad_sqnorm) or several partial sums (GEMM epilogue slots, per-chunk norms of a
        # data-parallel exchange) that the kernel adds up itself in a fixed order
        _req(sqnorm.dtype == torch.float32 and sqnorm.is_contiguous() and sqnorm.numel() >= 1,
             "sqnorm.dtype == torch.float32 and sqnorm.is_contiguous() and sqnorm.numel() >= 1")
        n_sq = sqnorm.numel()
    bc1 = 1.0 - beta1 ** step
    bc2 = 1.0 - beta2 ** step
    _count()
    c_dt = dtype_id(compact_out.dtype) if compact_out is not None else _lib.BF16
    w_dt = dtype_id(w_dtype) if w_dtype is not None else _lib.BF16
    with _timed("compact_adam", master.device, grad.numel()):
        check(load().smt_compact_adam(ptr(master), ptr(exp_avg), ptr(exp_avg_sq), ptr(grad), dtype_id(grad.dtype),
                                      grad.numel(), lr, beta1, beta2, eps, weight_decay, bc1, bc2, grad_scale,
                                      ptr(sqnorm), n_sq, max_norm, ptr(compact_out), c_dt, ptr(table), n_blocks, block,
                                      w_dt, _st(master)), "smt_compact_adam")



# ---- grouped block-gradient GEMM: several (x, dy) problems in one launch ------------------------------------

LAST_GROUP: dict = {}     # shape of the most recent grouped launch (bench.py reports it)
HOST_TIME = {"flush_s": 0.0, "flushes": 0, "operand_bytes_held_max": 0}   # host-side cost of grouped launches and the
                                                                           # bytes of x / dy kept alive until a flush (bench.py)

_ITEM_DT = None


def _item_dtype():
    global _ITEM_DT
    if _ITEM_DT is None:
        import numpy as np
        _ITEM_DT = np.dtype([("map_dy", "<u4"), ("map_x", "<u4"), ("row", "<i4"), ("col", "<i4"), ("out_off", "<i8"),
                             ("flags", "<u4"), ("sq_slot", "<i4")])
        assert _ITEM_DT.itemsize == C.sizeof(_lib.GemmItem) == 32
    return _ITEM_DT


class _Problem:
    __slots__ = ("x", "dy", "idx", "idx_id", "out", "block", "accumulate", "sq", "sq_slot0", "sink")

    def __init__(self, x, dy, idx, idx_id, out, block, accumulate, sq, sq_slot0, sink):
        self.x, self.dy, self.idx, self.idx_id, self.out, self.block = x, dy, idx, idx_id, out, block
        self.accumulate, self.sq, self.sq_slot0, self.sink = accumulate, sq, sq_slot0, sink


_idx_snap: dict = {}      # id(index_list) -> tuple snapshot (validated by value on every use)


def _snapshot_index_list(index_list):
    """Immutable ((row, col), ...) copy of a Python index list; the common case (same list object, same contents as
    last step) costs one tuple comparison instead of n int() conversions."""
    key = id(index_list)
    hit = _idx_snap.get(key)
    if hit is not None and len(hit) == len(index_list) and tuple(index_list) == hit:
        return hit
    snap = tuple((int(r), int(c)) for r, c in index_list)
    if len(_idx_snap) > 8192:
        _idx_snap.clear()
    _idx_snap[key] = snap
    return snap


class BlockGradBatch:
    """Collects block-gradient problems (one per module backward) and runs them as ONE grouped tcgen05 launch.

    add() keeps references to the operands; flush() encodes one TMA descriptor per distinct operand on the host,
    ships descriptors + per-block work items with a single pinned H2D copy and launches
    `smt_block_grad_gemm_grouped`.  Problems must share T, the input dtype, the output dtype and the block size
    (flush() launches one group per distinct combination).  The sorted / paired work-item array of a given set of
    problems is cached, so steady-state steps only re-encode the (pointer-dependent) TMA descriptors."""

    def __init__(self):
        self.problems = []
        self.last_flushed = []
        self._out_ptrs = set()
        self._plans: dict = {}

    def __len__(self):
        return len(self.problems)

    def n_blocks(self) -> int:
        return sum(len(pr.idx) for pr in self.problems)

    def add(self, x2d: torch.Tensor, dy2d: torch.Tensor, index_list, out: torch.Tensor, block: int,
            accumulate: bool = True, sq: Optional[torch.Tensor] = None, sq_slot0: int = -1, sink=None) -> None:
        """`accumulate=False`: this problem's blocks overwrite `out` (per-item flag) even though the launch as a whole
        accumulates.  `sq` / `sq_slot0`: fp32 tensor whose slots [sq_slot0 + 2 i, sq_slot0 + 2 i + 1] receive the sum
        of squares of block i as stored (when the launch shape supports it; `sink.sq_ok` is set accordingly)."""
        require_cuda(x2d, dy2d, out, sq)
        _req(x2d.dim() == 2 and dy2d.dim() == 2 and x2d.shape[0] == dy2d.shape[0] and x2d.dtype == dy2d.dtype,
             "x2d.dim() == 2 and dy2d.dim() == 2 and x2d.shape[0] == dy2d.shape[0] and x2d.dtype == dy2d.dtype")
        _req(x2d.stride(1) == 1 and dy2d.stride(1) == 1 and out.is_contiguous(),
             "x2d.stride(1) == 1 and dy2d.stride(1) == 1 and out.is_contiguous()")
        _req(out.numel() == len(index_list) * block * block, "out.numel() == len(index_list) * block * block")
        if out.data_ptr() in self._out_ptrs:
            # the same output twice in one launch would race (two tiles read-modify-write the same block)
            self.flush()
        self._out_ptrs.add(out.data_ptr())
        self.problems.append(_Problem(x2d, dy2d, _snapshot_index_list(index_list), id(index_list), out, int(block),
                                      bool(accumulate), sq, int(sq_slot0), sink))

    def flush(self, accumulate: bool = True) -> int:
        """Launches everything collected so far; returns the number of grouped launches.  `last_flushed` keeps the
        problems of this flush (their sinks have been updated)."""
        import time
        t0 = time.perf_counter()
        problems, self.problems = self.problems, []
        self._out_ptrs = set()
        held = {}
        for pr in problems:                                   # distinct operands this batch kept alive until now
            for t in (pr.x, pr.dy):
                held[t.data_ptr()] = t.shape[0] * t.stride(0) * t.element_size()
        HOST_TIME["operand_bytes_held_max"] = max(HOST_TIME["operand_bytes_held_max"], sum(held.values()))
        groups: dict = {}
        for pr in problems:
            if len(pr.idx) == 0 or pr.x.shape[0] == 0:
                continue
            key = (pr.x.shape[0], pr.x.dtype, pr.out.dtype, pr.block, pr.x.device,
                   pr.sq.data_ptr() if pr.sq is not None else 0)
            groups.setdefault(key, []).append(pr)
        for (T, in_dt, out_dt, block, dev, _sq), prs in groups.items():
            self._launch_group(T, in_dt, out_dt, block, dev, prs, accumulate)
        HOST_TIME["flush_s"] += time.perf_counter() - t0
        HOST_TIME["flushes"] += 1
        self.last_flushed = problems
        return len(groups)

    def _items_for(self, T, block, prs, maps_of, base_ptr, esize):
        """Work-item array for this set of problems (cached: index lists, output offsets and the sharing pattern of
        the operands do not change from step to step).
        Work-item order = execution order (CTAs / CTA pairs are dispatched in item order):
          * within a module, blocks are walked by (block row, block column), and two consecutive blocks of one block
            row form a PAIR: the cta_group::2 kernel gives items (2c, 2c+1) to CTA pair c and loads the shared dy strip
            once, so every pair must start at an even position;
          * a module's unpaired blocks follow its pairs immediately (their strips are still in L2), not at the end of
            the launch; an odd one out is carried over to the next module to keep the even alignment."""
        import numpy as np
        key = (T, block, tuple((pr.idx, (pr.out.data_ptr() - base_ptr) // esize, pr.accumulate,
                                pr.sq_slot0 if pr.sq is not None else -1, mx, mdy)
                               for pr, (mx, mdy) in zip(prs, maps_of)))
        hit = self._plans.get(key)
        if hit is not None:
            return hit
        items, carry = [], []
        for pr, (mx, mdy) in zip(prs, maps_of):
            off0 = (pr.out.data_ptr() - base_ptr) // esize
            flags = 0 if pr.accumulate else _lib.ITEM_OVERWRITE
            entries = [(mdy, mx, r, c, off0 + i * block * block, flags,
                        (pr.sq_slot0 + 2 * i) if (pr.sq is not None and pr.sq_slot0 >= 0) else -1)
                       for i, (r, c) in sorted(enumerate(pr.idx), key=lambda t: (t[1][0], t[1][1]))]
            pairs, singles, i = [], list(carry), 0
            while i < len(entries):
                if i + 1 < len(entries) and entries[i][2] == entries[i + 1][2]:
                    pairs += [entries[i], entries[i + 1]]
                    i += 2
                else:
                    singles.append(entries[i])
                    i += 1
            carry = [singles.pop()] if len(singles) % 2 else []
            items += pairs + singles
        items += carry
        arr = np.array(items, dtype=_item_dtype())
        n_pairs = sum(1 for k in range(0, len(items) - 1, 2)
                      if items[k][0] == items[k + 1][0] and items[k][2] == items[k + 1][2])
        if len(self._plans) > 64:
            self._plans.clear()
        self._plans[key] = (arr, n_pairs)
        return arr, n_pairs

    def _launch_group(self, T, in_dt, out_dt, block, dev, prs, accumulate) -> None:
        lib = load()
        maps: dict = {}

        def map_index(t: torch.Tensor) -> int:
            key = (t.data_ptr(), t.shape[1], t.stride(0))
            if key not in maps:
                maps[key] = (len(maps), t)
            return maps[key][0]

        esize = prs[0].out.element_size()
        base_ptr = min(pr.out.data_ptr() for pr in prs)
        maps_of = [(map_index(pr.x), map_index(pr.dy)) for pr in prs]
        arr, n_pairs = self._items_for(T, block, prs, maps_of, base_ptr, esize)
        n_items, n_maps = len(arr), len(maps)
        sq = prs[0].sq
        emits = bool(sq is not None and lib.smt_block_grad_gemm_grouped_emits_sq(n_items, block, T))
        LAST_GROUP.update(items=n_items, operands=n_maps,
                          cta_group_2=bool(lib.smt_block_grad_gemm_grouped_uses_2sm(n_items, block, T)),
                          row_sharing_pairs=n_pairs, emits_sq=emits)
        nbytes = n_maps * 128 + arr.nbytes
        stage = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        host = stage.numpy()
        in_id = dtype_id(in_dt)
        for _key, (i, t) in maps.items():
            check(lib.smt_encode_operand_map(stage.data_ptr() + i * 128, t.data_ptr(), t.shape[1], T, t.stride(0),
                                             in_id, block), "smt_encode_operand_map")
        host[n_maps * 128:] = arr.view("u1").reshape(-1)
        dev_buf = stage.to(dev, non_blocking=True)
        ws_bytes = lib.smt_block_grad_gemm_grouped_workspace_bytes(n_items, block, T)
        ws = _workspace(ws_bytes, dev)
        with _timed("block_grad_gemm", dev, (n_items, block, T)):
            check(lib.smt_block_grad_gemm_grouped(dev_buf.data_ptr(), dev_buf.data_ptr() + n_maps * 128, n_items,
                                                  T, block, in_id, base_ptr, dtype_id(out_dt), 1 if accumulate else 0,
                                                  0, ptr(sq) if emits else 0, ptr(ws), ws_bytes, stream_ptr(dev)),
                  "smt_block_grad_gemm_grouped")
        _count(lib.smt_last_launch_count())
        for pr in prs:
            if pr.sink is not None:
                pr.sink.sq_ok = emits
