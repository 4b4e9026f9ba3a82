"""Drop-in mirror of the reference module `deepspeed/smt/smt.py`, backed by sm_100a kernels.

Public names kept identical to what the reference driver imports (fine_tune.py:39):

    LinearLayer_MatrixSparsity                smt.py:302-344
    linearZ                                   smt.py:347-413
    convert_linear_layer_to_matrix_sparsity   smt.py:83-179
    convert_matrix_sparsity_to_linear_layer   smt.py:416-457
    freeze_unselected_matrix_layer            smt.py:641-745
    get_optimizer_sparse_grouped_parameters   smt.py:465-549
    get_optimizer_qk_augment_grouped_parameters  smt.py:554-638
    Block_dimension                           smt.py:22 (module global, read at call time)

What changed underneath:
  * `__init__` gathers all selected blocks with ONE kernel launch (`smt_block_gather`) instead of n slice copies;
  * `forward` scatters compact -> dense with ONE launch on every call, exactly when the reference does
    (smt.py:332-341; it issues n slice copies).  The only case in which the launch is skipped is when the fused
    optimizer (`SMTAdam`) has itself written the updated blocks into the dense weight and says so (`mark_synced`);
    any optimizer that updates `selected_weight` behind our back (DeepSpeed FusedAdam through `p.data`, ZeRO flat
    partitions) therefore always sees its update in the next forward;
  * `linearZ.backward` forms every selected block gradient in ONE grouped tcgen05/TMEM GEMM
    (`smt_block_grad_gemm`): fp32 accumulation over all B*S tokens, rounded once — the reference does a bmm, a
    batch reduction and a slice copy per block, rounding to bf16 per batch entry;
  * importing this module does not call `deepspeed.init_distributed()` (the reference does, smt.py:20).

The channel-sparsity twins (`LinearLayer_ChannelSparsity`, `linearChannel`, `convert_linear_layer_to_channel_sparsity`,
`freeze_unselected_channel_layer`; smt.py:25-80, 185-296, 748-831) keep the reference's names and signatures but use
COLUMN semantics: the reference selects input channels, differentiates weight columns and copies weight rows, which
fails for every non-square weight (SURVEY.md section 2 row 16).  Its gradient formula is kept exactly.
"""
from __future__ import annotations

import contextlib
import re
import threading
import warnings
import weakref
from typing import Dict, Tuple

import torch
from torch import nn

from .. import decoder_fusion, ops
from .._lib import SMTLibraryError

Block_dimension = 256

_LAYER_RE = re.compile(r"model\.layers\.(\d+)\.")
_MLP_NAMES = ("gate_proj", "up_proj", "down_proj")
_ATTN_NAMES = ("q_proj", "k_proj", "v_proj", "o_proj")


def _rank0_print(msg: str) -> None:
    if not torch.distributed.is_available() or not torch.distributed.is_initialized() \
            or torch.distributed.get_rank() == 0:
        print(msg)


def _getattr_path(root, dotted: str):
    obj = root
    for part in dotted.split("."):
        obj = getattr(obj, part)
    return obj


def _setattr_path(root, dotted: str, value) -> None:
    parts = dotted.split(".")
    obj = root
    for part in parts[:-1]:
        obj = getattr(obj, part)
    setattr(obj, parts[-1], value)


def _layer_of(name: str):
    m = _LAYER_RE.search(name)
    return int(m.group(1)) if m else None


def _mlp_kind(name: str) -> str:
    # smt.py:104 — anything that is not gate/up falls through to 'down_proj'
    return "gate_proj" if "gate_proj" in name else "up_proj" if "up_proj" in name else "down_proj"


def _attn_kind(name: str):
    # smt.py:120 — q, k, v, o by substring, else None
    for kind in _ATTN_NAMES:
        if kind in name:
            return kind
    return None


# ---- device-side index tables ---------------------------------------------------------------------------

_rc_cache: Dict[Tuple[int, torch.device], Tuple[tuple, torch.Tensor]] = {}


def _block_rc_for(index_list, device) -> torch.Tensor:
    """int32 [n, 2] device copy of a Python index list, cached per list object and validated by value
    (linearZ receives only the plain list, exactly like the reference)."""
    snap = tuple((int(r), int(c)) for r, c in index_list)
    key = (id(index_list), device)
    hit = _rc_cache.get(key)
    if hit is not None and hit[0] == snap:
        return hit[1]
    t = ops.make_block_rc(snap, device)
    if len(_rc_cache) > 4096:
        _rc_cache.clear()
    _rc_cache[key] = (snap, t)
    return t


# ---- deferred, grouped block-gradient launches (native mode only) ------------------------------------------------
#
# With a gradient sink (SMTAdam's flat buffer) nothing has to be RETURNED by linearZ.backward, so the contraction can
# be postponed: every module's backward only enqueues its (x, dy, blocks, sink) problem (linearChannel: its
# (partial, dy, n, sink) problem, whose tiles are stored with the row pitch out_features) and ONE grouped tcgen05
# launch runs when the autograd engine finishes the backward pass (a queue_callback), i.e. before
# `loss.backward()` returns.  Per-module launches of ~9-30 blocks cannot fill 148 SMs; the grouped launch of all
# 869 blocks can.  `flush_block_grads()` is also called by SMTAdam.step() / dp.allreduce_compact_grads as a guard.

_grouped = {"enabled": False, "chunk_blocks": 0}
_pending = ops.BlockGradBatch()
_pending_lock = threading.Lock()
_pending_state = {"callback_queued": False, "stream": None, "last_x": None}
_flush_listeners = []


def set_grouped_backward(enabled: bool, chunk_blocks: int = 0) -> None:
    """Enable / disable deferral of the block-gradient GEMMs to grouped launches.

    chunk_blocks = 0: ONE launch per backward pass (when the autograd engine finishes).
    chunk_blocks > 0: additionally flush DURING the backward pass, at a layer boundary (a module with a different
    input arrives), whenever at least that many blocks are pending - each chunk still fills the GPU (choose >= 148
    tiles) and a data-parallel exchange can all-reduce it while the rest of the backward pass runs (dp.py).
    Measured on 2 / 8 B200 (profiles/r02_scaling_breakdown.md): ~192 (three chunks of the 869-block selection) is the
    sweet spot - the NCCL kernels only get SMs in the gaps between the backward pass's kernels, so chunks must be
    flushed EARLY to be reduced by the time backward ends; two big chunks (284 / 504) left 1.4-2.7 ms exposed, three
    small ones 0.3 ms, at the price of one more 0.1 ms round of the GEMM."""
    flush_block_grads()
    _grouped["enabled"] = bool(enabled)
    _grouped["chunk_blocks"] = int(chunk_blocks) if enabled else 0


def add_flush_listener(fn) -> None:
    """`fn(sinks)` is called after every grouped launch with the GradSinks it delivered to (on the thread and the
    stream that launched it)."""
    if fn not in _flush_listeners:
        _flush_listeners.append(fn)


def remove_flush_listener(fn) -> None:
    if fn in _flush_listeners:
        _flush_listeners.remove(fn)


def _flush_locked() -> int:
    if len(_pending) == 0:
        return 0
    stream = _pending_state["stream"]
    ctx = torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()
    with ctx:
        launches = _pending.flush(accumulate=True)
        sinks = [pr.sink for pr in _pending.last_flushed if pr.sink is not None]
        for fn in list(_flush_listeners):
            fn(sinks)
    return launches


def flush_block_grads() -> int:
    """Run every pending block-gradient problem now (no-op when nothing is pending)."""
    with _pending_lock:
        _pending_state["callback_queued"] = False
        _pending_state["last_x"] = None
        return _flush_locked()


def _enqueue(xkey, device, add) -> None:
    """Queue one module's gradient problem (`add()` puts it into `_pending`); `xkey` identifies the module's input, so
    that a chunked flush happens at a layer boundary."""
    with _pending_lock:
        chunk = _grouped["chunk_blocks"]
        if chunk > 0 and _pending_state["last_x"] not in (None, xkey) and _pending.n_blocks() >= chunk:
            _flush_locked()                                     # layer boundary with a GPU-filling chunk pending
        _pending_state["last_x"] = xkey
        add()
        _pending_state["stream"] = torch.cuda.current_stream(device)
        if not _pending_state["callback_queued"]:
            _pending_state["callback_queued"] = True
            torch.autograd.Variable._execution_engine.queue_callback(flush_block_grads)


def _enqueue_block_grad(x2, dy2, index_list, sink, block, accumulate) -> None:
    _enqueue((x2.data_ptr(), x2.shape[0]), x2.device,
             lambda: _pending.add(x2, dy2, index_list, sink.view, block, accumulate=accumulate, sq=sink.sq,
                                  sq_slot0=sink.sq_slot0, sink=sink))


class linearZ(torch.autograd.Function):
    """y = x W^T with a block-sparse weight gradient.  Reference: smt.py:347-413.

    forward(ctx, input, selected_weight, matrix_index_list, weight)
    backward -> (grad_input, grad_weight [n*b, b], None, None)
    """

    @staticmethod
    def forward(ctx, input, selected_weight, matrix_index_list, weight):
        ctx.block = Block_dimension
        ctx.index_list = matrix_index_list
        ctx.sw_ref = selected_weight                      # only for the optional gradient sink (no data use)
        ctx.save_for_backward(input, weight)              # the reference keeps column views of `input` alive
        return torch.matmul(input, weight.t())            # smt.py:366 (dense, cuBLAS)

    @staticmethod
    def backward(ctx, grad_output):
        x, weight = ctx.saved_tensors
        grad_input = grad_weight = None
        if ctx.needs_input_grad[1]:
            x2 = _as_operand(x.reshape(-1, x.shape[-1]))
            dy2 = _as_operand(grad_output.reshape(-1, grad_output.shape[-1]))
            grad_weight = _block_weight_grad(ctx.sw_ref, ctx.index_list, x2, dy2, ctx.block, grad_output.dtype)
        if ctx.needs_input_grad[0]:
            grad_input = torch.matmul(grad_output, weight)                                      # smt.py:406
        return grad_input, grad_weight, None, None


def _as_operand(t2):
    """[T, features] view usable by TMA: unit column stride, 16-byte row pitch and base."""
    if t2.stride(-1) != 1 or (t2.stride(0) * t2.element_size()) % 16 != 0 or t2.data_ptr() % 16 != 0:
        t2 = t2.contiguous()
    return t2


def _block_weight_grad(sw_param, index_list, x2, dy2, b, out_dtype):
    """The block gradients of one module (smt.py:382-404).  Native mode (the parameter owns a GradSink, i.e. it lives
    in an SMTAdam arena): delivered straight into the flat gradient buffer - grouped with the other modules of the
    backward pass when grouping is enabled - and None is returned; otherwise the [n*b, b] gradient is returned."""
    n = len(index_list)
    if x2.dtype != dy2.dtype:
        x2 = x2.to(dy2.dtype)
    sink = getattr(sw_param, "_smt_sink", None)
    if sink is not None:
        # the sink says whether this delivery accumulates or overwrites (first one after a lazy zero_grad)
        accumulate = sink.begin_delivery(sw_param)
        if _grouped["enabled"] and dy2.dtype != torch.float32 and n > 0:
            _enqueue_block_grad(x2, dy2, index_list, sink, b, accumulate)   # grouped launch(es) per backward
        else:
            rc = _block_rc_for(index_list, dy2.device)
            ops.block_grad_gemm(x2, dy2, rc, b, out=sink.view, accumulate=accumulate, index_list=index_list)
            sink.sq_ok = False
        return None
    rc = _block_rc_for(index_list, dy2.device)
    return ops.block_grad_gemm(x2, dy2, rc, b, out_dtype=out_dtype, index_list=index_list).view(n * b, b)   # smt.py:382-404


class LinearLayer_MatrixSparsity(nn.Module):
    """Linear layer whose only trainable parameter is a compact copy of its selected b x b blocks.
    Reference: smt.py:302-344 (same constructor signature and attribute names)."""

    def __init__(self, weight, bias=None, index_list=[]):
        super().__init__()
        if not weight.is_cuda:
            raise SMTLibraryError("LinearLayer_MatrixSparsity needs its weight on a CUDA device: the SMT kernels "
                                  "have no CPU fallback")
        b = Block_dimension
        self.weight = weight
        self.weight.requires_grad = False                 # smt.py:308
        self.bias = bias                                  # kept but unused, exactly like smt.py:309,343
        self.index_list = index_list
        self.block = b
        for (r, c) in index_list:
            if not (0 <= r < weight.shape[0] // b and 0 <= c < weight.shape[1] // b):
                raise IndexError(f"block ({r}, {c}) outside a {tuple(weight.shape)} weight with block {b}")
        n = len(index_list)
        compact = torch.empty(n * b, b, dtype=weight.dtype, device=weight.device)
        self._table = None
        self._table_key = None
        if n:
            ops.block_gather(self._block_table(), n, b, compact)       # smt.py:317-325
        self.selected_weight = nn.Parameter(compact, requires_grad=True)
        self.selected_weight._smt_owner = weakref.ref(self)   # lets SMTAdam find the dense weight to write back
        self.fn = linearZ.apply
        # Set ONLY by `mark_synced()` (= SMTAdam after its fused write-back): (storage pointer, version) of
        # selected_weight at that moment.  None = "nobody vouches for the dense weight": scatter on every forward.
        self._synced = None

    # -- device table of (W pointer, ld, row, col) per block, rebuilt if the weight storage moves --
    def _block_table(self) -> torch.Tensor:
        w = self.weight.data
        key = (w.data_ptr(), w.stride(0), w.device)
        if self._table is None or self._table_key != key:
            self._table = ops.make_block_table([(w, r, c) for r, c in self.index_list], w.device)
            self._table_key = key
        return self._table

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._table = None
        self._synced = None
        return out

    # -- what SMTAdam's arena (optim._Arena) asks of the layer that owns a parameter --
    def _arena_ok(self) -> bool:
        return True

    def _arena_layout(self):
        """(elements the arena reserves for selected_weight, sum-of-squares slots its gradient launches fill)"""
        n = len(self.index_list)
        return n * self.block * self.block, 2 * n

    def _writeback(self, off: int):
        """(key, entries) of the dense write-back of selected_weight stored at arena offset `off`: owners with equal keys
        share one fused Adam launch, whose table `_writeback_args` builds from their concatenated entries."""
        return ("blocks", self.block, self.weight.dtype), [(self.weight.data, r, c) for r, c in self.index_list]

    @staticmethod
    def _writeback_args(key, entries, device) -> dict:
        return dict(table=ops.make_block_table(entries, device), n_blocks=len(entries), block=key[1], w_dtype=key[2])

    def mark_synced(self) -> None:
        """Called by the fused optimizer (SMTAdam) right after it has written the updated blocks into `weight`
        itself.  The mark is tied to the parameter's storage pointer and version counter: re-pointing `.data`
        (DeepSpeed / ZeRO flat buffers) or any version-counted write to the Parameter invalidates it.  Writes
        through `selected_weight.data` are invisible to the version counter, so whoever does that while SMTAdam
        owns the parameter must call `sync_weight(force=True)`; without SMTAdam nothing is ever skipped."""
        self._synced = (self.selected_weight.data_ptr(), self.selected_weight._version)

    def sync_weight(self, force: bool = False) -> None:
        """compact -> dense write-back (smt.py:332-341): ONE launch per call.  Unconditional like the reference's
        loop, except right after an SMTAdam step that wrote the dense blocks itself (see `mark_synced`)."""
        if not force and self._synced is not None and \
                self._synced == (self.selected_weight.data_ptr(), self.selected_weight._version):
            return
        self._synced = None
        n = len(self.index_list)
        if n:
            sw = self.selected_weight.data
            if sw.dtype != self.weight.dtype:
                sw = sw.to(self.weight.dtype)
            ops.block_scatter(self._block_table(), n, self.block, sw.contiguous())

    def forward(self, x):
        self.sync_weight()
        return self.fn(x, self.selected_weight, self.index_list, self.weight)   # smt.py:343


# ---- fused q/k/v projections (SURVEY section 8f row 2: the dense side of linearZ) --------------------------------
#
# q_proj, k_proj and v_proj of a decoder layer read the same hidden states.  The reference runs them as three
# independent modules: three `x @ W^T` GEMMs in forward (smt.py:366), three `dy @ W` GEMMs in backward (smt.py:406) whose
# results autograd adds with two elementwise kernels.  `fuse_qkv_projections(model)` ties the three modules of every
# layer into a group: the first call (q_proj) runs ONE hand-written tcgen05 GEMM over [Wq; Wk; Wv] and hands k_proj /
# v_proj their slices when they are called with the same tensor; backward runs ONE GEMM over K = 4096 + 1024 + 1024
# for the input gradient and feeds the weight-gradient path of each sparse member.  Module names, parameters and
# state dicts are untouched (the override is a method bound to the instance); members may be LinearLayer_MatrixSparsity,
# bf16 LinearLayer_ChannelSparsity or frozen, bias-free nn.Linear.  Anything the kernel does not support falls back to
# the members' own forward.
# The same call also moves the layer's elementwise ops (norms, residual add, RoPE, SwiGLU) onto native kernels
# (decoder_fusion.py).

class fusedLinearZ(torch.autograd.Function):
    """forward(ctx, input, group, *selected_weights of the sparse members) -> one output per member.
    Block members keep `input` for their gradient; channel members keep only their packed input channels (linearChannel)."""

    @staticmethod
    def forward(ctx, input, group, *selected_weights):
        weights = [m.weight for m in group.members]
        x2 = _as_operand(input.reshape(-1, input.shape[-1]))
        ys = ops.fused_linear_forward(x2, [w.data for w in weights])
        ctx.group = group
        ctx.block = Block_dimension
        ctx.x_shape = input.shape
        ctx.xkey = (x2.data_ptr(), x2.shape[0])
        partials = []
        sparse = [m for m in group.members if isinstance(m, _SPARSE_LAYERS)]
        for k, m in enumerate(sparse):
            if isinstance(m, LinearLayer_ChannelSparsity):
                partials.append(ops.channel_gather(x2, _channel_idx_for(m.index_list, x2.device, 8))
                                if ctx.needs_input_grad[2 + k] and len(m.index_list) else None)   # smt.py:240-247
        keep_x = any(isinstance(m, LinearLayer_MatrixSparsity) for m in sparse)
        ctx.n_partials = len(partials)
        ctx.save_for_backward(input if keep_x else None, *partials, *weights)
        lead = input.shape[:-1]
        return tuple(y.view(*lead, y.shape[-1]) for y in ys)

    @staticmethod
    def backward(ctx, *grad_outputs):
        x, *saved = ctx.saved_tensors
        partials, weights = saved[:ctx.n_partials], saved[ctx.n_partials:]
        members = ctx.group.members
        dys = [_as_operand(g.reshape(-1, g.shape[-1])) for g in grad_outputs]
        grad_input = None
        if ctx.needs_input_grad[0]:
            grad_input = ops.fused_linear_dgrad(dys, [w.data for w in weights]).view(ctx.x_shape)   # smt.py:406, all members
        grads, k, j = [], 0, 0
        x2 = None
        for m, dy2 in zip(members, dys):
            if not isinstance(m, _SPARSE_LAYERS):
                continue
            g = None
            if isinstance(m, LinearLayer_ChannelSparsity):
                partial = partials[j]
                j += 1
                if ctx.needs_input_grad[2 + k]:
                    g = _channel_weight_grad(m.selected_weight, partial, len(m.index_list), dy2, ctx.xkey)
            elif ctx.needs_input_grad[2 + k]:
                if x2 is None:
                    x2 = _as_operand(x.reshape(-1, x.shape[-1]))
                g = _block_weight_grad(m.selected_weight, m.index_list, x2, dy2, ctx.block, dy2.dtype)
            grads.append(g)
            k += 1
        return (grad_input, None, *grads)


class _SharedInputGroup:
    """q_proj / k_proj / v_proj of one attention layer, in call order."""

    def __init__(self, members):
        self.members = list(members)
        self._cache = None           # (input tensor, [outputs still to be handed out])
        self._ok_key = None

    def _supported(self, x) -> bool:
        ws = [m.weight for m in self.members]
        if not (x.is_cuda and x.dim() >= 2 and x.dtype == ws[0].dtype and x.shape[-1] == ws[0].shape[1]):
            return False
        key = tuple((w.data_ptr(), w.stride(0), w.dtype) for w in ws)
        if self._ok_key != key:
            ok = ops.fused_linear_supported([w.data for w in ws], dgrad=False) and \
                ops.fused_linear_supported([w.data for w in ws], dgrad=True)
            self._ok_key = key if ok else None
            if not ok:
                return False
        return True

    def call(self, role: int, module, x):
        c = self._cache
        if role != 0 and c is not None and c[0] is x and c[1][role] is not None:
            y, c[1][role] = c[1][role], None
            if all(o is None for o in c[1]):
                self._cache = None
            return y
        if role == 0 and self._supported(x):
            sparse = [m for m in self.members if isinstance(m, _SPARSE_LAYERS)]
            for m in sparse:
                m.sync_weight()                         # smt.py:332-341 / 208-211, unless SMTAdam vouches
            outs = list(fusedLinearZ.apply(x, self, *[m.selected_weight for m in sparse]))
            y, outs[0] = outs[0], None
            self._cache = (x, outs)
            return y
        return type(module).forward(module, x)                         # different input / unsupported: the plain path


def _fusable_member(m) -> bool:
    if isinstance(m, LinearLayer_MatrixSparsity):
        return True
    if isinstance(m, LinearLayer_ChannelSparsity):
        return m.weight.dtype == torch.bfloat16 and m.selected_weight.dtype == torch.bfloat16
    return isinstance(m, nn.Linear) and m.bias is None and not m.weight.requires_grad


def _shared_group_forward(self, x):
    return self._smt_shared_group.call(self._smt_group_role, self, x)


def fuse_qkv_projections(model) -> int:
    """Fuses the dense-side work of every decoder layer it can: q_proj / k_proj / v_proj of each attention module become
    one fused dense GEMM per direction (see above), and in a LLaMA, Mistral or Qwen3 decoder layer whose projections
    were fused the elementwise ops around them - the two RMSNorms with the residual add, RoPE (with Qwen3's per-head
    q/k norms) and SwiGLU - run on the native kernels of
    `decoder_fusion` (the model's final norm too).  Returns the number of layers whose projections were fused.  Call
    after `convert_linear_layer_to_matrix_sparsity` / `convert_linear_layer_to_channel_sparsity`; undone by
    `unfuse_qkv_projections` (and automatically by `convert_matrix_sparsity_to_linear_layer` /
    `convert_channel_sparsity_to_linear_layer`).  The overrides are methods bound to each module, so a `copy.deepcopy`
    of the model computes with the copy's weights."""
    fused = 0
    for parent in model.modules():
        trio = [getattr(parent, n, None) for n in ("q_proj", "k_proj", "v_proj")]
        if any(t is None for t in trio) or not all(_fusable_member(t) for t in trio):
            continue
        if any(getattr(t, "_smt_shared_group", None) is not None for t in trio):
            continue
        ws = [t.weight for t in trio]
        if not all(w.is_cuda for w in ws) or not ops.fused_linear_supported([w.data for w in ws], dgrad=False) \
                or not ops.fused_linear_supported([w.data for w in ws], dgrad=True):
            continue
        group = _SharedInputGroup(trio)
        for role, mod in enumerate(trio):
            mod._smt_shared_group = group
            mod._smt_group_role = role
            decoder_fusion.install_forward(mod, _shared_group_forward)
        fused += 1
    layers = [m for m in model.modules() if getattr(getattr(getattr(m, "self_attn", None), "q_proj", None),
                                                   "_smt_shared_group", None) is not None]
    n_elementwise = sum(decoder_fusion.install_layer(m) for m in layers)
    if n_elementwise:
        for m in model.modules():
            if isinstance(getattr(m, "layers", None), nn.ModuleList) and any(l in layers for l in m.layers):
                decoder_fusion.install_norm(getattr(m, "norm", None))
    if n_elementwise < len(layers):
        warnings.warn(f"fuse_qkv_projections: elementwise ops of {len(layers) - n_elementwise} of {len(layers)} decoder "
                      "layers left to transformers (not a LLaMA, Mistral or Qwen3 decoder layer of the supported "
                      "transformers version, head_dim 128, SiLU)")
    return fused


def unfuse_qkv_projections(model) -> int:
    """Restores every module `fuse_qkv_projections` touched to its class's own forward; returns the number of q/k/v
    groups undone."""
    n = 0
    for mod in model.modules():
        if getattr(mod, "_smt_shared_group", None) is not None:
            decoder_fusion.remove_forward(mod)
            mod.__dict__.pop("_smt_shared_group", None)
            mod.__dict__.pop("_smt_group_role", None)
            n += 1
    decoder_fusion.remove_all(model)
    return n // 3


def fuse_causal_lm_loss(model) -> bool:
    """Runs the lm_head and causal-LM cross-entropy of a `LlamaForCausalLM`, `MistralForCausalLM` or `Qwen3ForCausalLM`
    as one chunked native op that never builds the fp32 logits (`decoder_fusion.LinearCrossEntropyFn`).  It applies to
    training calls with `labels` (grad mode on, `logits_to_keep=0`, no KV cache, CUDA bf16, a frozen bias-free lm_head
    with `out_features == vocab_size`, a vocabulary that is a multiple of 64 and at least 256); those
    return the loss with `logits=None`.  `shift_labels`, `ignore_index` and `num_items_in_batch` are honoured as
    transformers' `ForCausalLMLoss` honours them.  Every other call runs the class's own forward, so evaluation under
    `no_grad` still gets logits.  Returns False (and changes nothing) for any other model class.  The override is a
    method bound to the model, so a `copy.deepcopy` computes with the copy's weights; undone by
    `unfuse_causal_lm_loss`."""
    return decoder_fusion.install_causal_lm(model)


def unfuse_causal_lm_loss(model) -> bool:
    """Restores the class's own forward on a model `fuse_causal_lm_loss` touched; False when there was nothing to undo."""
    return decoder_fusion.remove_causal_lm(model)


# ---- model surgery ---------------------------------------------------------------------------------------

def _selection_key_and_table(name: str, mixture: bool, selected_submatrix, selected_submatrix_attention):
    """Which (module, layer) key and which selection dict a Linear called `name` is looked up in.
    Mirrors the branch structure of smt.py:98-176."""
    if "mlp" in name:
        return (_mlp_kind(name), _layer_of(name)), selected_submatrix
    if "self_attn" in name:
        table = selected_submatrix if mixture else selected_submatrix_attention
        return (_attn_kind(name), _layer_of(name)), table
    if mixture and "embed_tokens" in name:
        return ("embed_tokens", None), selected_submatrix
    return None, None


def convert_linear_layer_to_matrix_sparsity(model,
                                            selected_submatrix,
                                            selected_submatrix_attention,
                                            part_module_name=['.layers'],
                                            mixture=False):
    """Reference: smt.py:83-179.  Every nn.Linear under `part_module_name` whose weight still requires grad
    (i.e. survived `freeze_unselected_matrix_layer`) becomes a LinearLayer_MatrixSparsity; bias is dropped
    (smt.py:113-115); layers without a selected block stay frozen nn.Linear."""
    names = [name for name, module in model.named_modules()
             if isinstance(module, nn.Linear) and any(part in name for part in part_module_name)]
    for name in names:
        key, table = _selection_key_and_table(name, mixture, selected_submatrix, selected_submatrix_attention)
        if key is None:
            continue
        module = _getattr_path(model, name)
        if not module.weight.requires_grad:
            continue
        _rank0_print(f"Module Test: {name}")
        index_list = table[key]                            # KeyError here = the reference's behaviour too
        sparse = LinearLayer_MatrixSparsity(module.weight, bias=None, index_list=index_list)
        _setattr_path(model, name, sparse.to(module.weight.device).to(module.weight.dtype))
    return model


def convert_matrix_sparsity_to_linear_layer(model, part_module_name=['.layers']):
    """Reference: smt.py:416-457: write the trained blocks back and restore plain nn.Linear modules that
    share the (now merged) weight Parameter."""
    unfuse_qkv_projections(model)
    names = [name for name, module in model.named_modules()
             if isinstance(module, LinearLayer_MatrixSparsity) and any(part in name for part in part_module_name)]
    for name in names:
        module = _getattr_path(model, name)
        module.sync_weight(force=True)
        out_f, in_f = module.weight.shape
        linear = nn.Linear(in_f, out_f, bias=False, device="meta")
        linear = linear.to_empty(device=module.weight.device).to(module.weight.dtype)
        linear.weight = module.weight                      # smt.py:451 — same Parameter, no clone
        _setattr_path(model, name, linear)
    return model


def freeze_unselected_matrix_layer(model,
                                   select_parameters,
                                   select_attention_parameters,
                                   mixture=False,
                                   layernorm=False):
    """Reference: smt.py:641-745.  requires_grad is True exactly for the parameters of modules that own a
    selected block (plus layer norms in mixture+layernorm mode); everything else is frozen."""
    for name, param in model.named_parameters():
        layer = _layer_of(name)
        if "mlp" in name:
            trainable = (_mlp_kind(name), layer) in select_parameters.keys()
        elif "self_attn" in name:
            table = select_parameters if mixture else select_attention_parameters
            trainable = (_attn_kind(name), layer) in table.keys()
        elif mixture and "embed_tokens" in name:
            trainable = ("embed_tokens", None) in select_parameters.keys()
        elif mixture and ("input_layernorm" in name or "post_attention_layernorm" in name):
            trainable = bool(layernorm)
        else:
            trainable = False
        param.requires_grad = trainable
    return model


def _grouped_parameters(model, weight_decay, base_lr, special_lr, no_decay_name_list, special_name_list):
    decay, special, no_decay = [], [], []
    for n, p in model.named_parameters():
        if not p.requires_grad:
            continue
        low = n.lower()
        if any(nd in low for nd in no_decay_name_list):
            no_decay.append((n, p))
        elif any(sp in low for sp in special_name_list):
            special.append((n, p))
        else:
            decay.append((n, p))
    for tag, items in (("0", decay), ("1", special), ("2", no_decay)):
        _rank0_print(f"================ PRINT PARAM NAME [{tag}]=======================")
        for n, _p in items:
            _rank0_print(f"name{tag}:{n}")
    groups = [
        {"params": [p for _n, p in decay], "weight_decay": weight_decay, "lr": base_lr},
        {"params": [p for _n, p in special], "weight_decay": weight_decay, "lr": special_lr},
        {"params": [p for _n, p in no_decay], "weight_decay": 0.0},
    ]
    return [g for g in groups if g["params"]]


def get_optimizer_sparse_grouped_parameters(
    model,
    weight_decay,
    smt_lr,
    lora_lr=5e-4,
    no_decay_name_list=["bias", "layer_norm.weight", "layernorm.weight", "norm.weight", "ln_f.weight"],
    lora_name_list=["lora_right_weight", "lora_left_weight"],
):
    """Reference: smt.py:465-549. Group 0 carries lr=smt_lr (it overrides the optimizer's lr); empty groups
    are dropped, so in practice one group holds every `selected_weight`."""
    return _grouped_parameters(model, weight_decay, smt_lr, lora_lr, no_decay_name_list, lora_name_list)


def get_optimizer_qk_augment_grouped_parameters(
    model,
    weight_decay,
    ft_learning_rate,
    module_lr=5e-4,
    no_decay_name_list=["bias", "layer_norm.weight", "layernorm.weight", "norm.weight", "ln_f.weight"],
    module_name_list=["q_proj", "k_proj"],
):
    """Reference: smt.py:554-638 (a full-fine-tuning option of the driver, fine_tune.py:160-163)."""
    return _grouped_parameters(model, weight_decay, ft_learning_rate, module_lr, no_decay_name_list,
                               module_name_list)


# ---- channel sparsity (SURVEY section 8f row 4: the activation-selected path, done consistently) -----------------
#
# The reference's LinearLayer_ChannelSparsity (smt.py:185-296) is selected by INPUT-channel activation scores
# (smt_helper.py:149-230), computes the gradient of weight COLUMNS `partial_input^T @ grad_output` (smt.py:283-284)
# but initialises from and writes back to weight ROWS (smt.py:198-200, 208-211): it fails for every non-square weight
# and trains the wrong entries for square ones.  Here channel i owns COLUMN index_list[i] of W; `selected_weight` is
# [n, out_features] (row i = W[:, index_list[i]]), so the gradient formula is the reference's, bit for bit in fp32.

_idx_cache: Dict[Tuple[int, torch.device], Tuple[tuple, torch.Tensor]] = {}


def _channel_idx_for(index_list, device, pad_to: int = 1) -> torch.Tensor:
    """int32 device copy of a channel index list (cached per list object, validated by value); `pad_to` > 1 appends -1
    entries ("zero column") up to a multiple of it."""
    snap = tuple(int(i) for i in index_list)
    key = (id(index_list), device, pad_to)
    hit = _idx_cache.get(key)
    if hit is not None and hit[0] == snap:
        return hit[1]
    t = ops.make_channel_idx(snap, device, pad_to)
    if len(_idx_cache) > 4096:
        _idx_cache.clear()
    _idx_cache[key] = (snap, t)
    return t


class linearChannel(torch.autograd.Function):
    """y = x W^T with a gradient only for the selected input channels.  Reference: smt.py:220-296.

    forward(ctx, input, selected_weight, channel_index_list, weight)
    backward -> (grad_input, grad_weight [n, out_features], None, None)
    """

    @staticmethod
    def forward(ctx, input, selected_weight, channel_index_list, weight):
        x2 = input.reshape(-1, input.shape[-1])
        if x2.stride(-1) != 1:
            x2 = x2.contiguous()
        # packed copy of the selected input channels, ONE launch (smt.py:240-247 does n strided slice copies); padded
        # with zero columns so that the tcgen05 gradient kernel can read it through TMA (16-byte row pitch) - fp32 inputs
        # take the fp32 block kernel, which wants whole 64-column blocks
        pad = 64 if x2.dtype == torch.float32 else 8
        partial = ops.channel_gather(x2, _channel_idx_for(channel_index_list, x2.device, pad))
        ctx.n_channels = len(channel_index_list)
        ctx.sw_ref = selected_weight                      # only for the optional gradient sink (no data use)
        ctx.xkey = (x2.data_ptr(), x2.shape[0])
        ctx.save_for_backward(partial, weight)
        return torch.matmul(input, weight.t())            # smt.py:257

    @staticmethod
    def backward(ctx, grad_output):
        partial, weight = ctx.saved_tensors
        grad_input = grad_weight = None
        if ctx.needs_input_grad[1]:
            dy2 = grad_output.reshape(-1, grad_output.shape[-1])
            if dy2.stride(-1) != 1 or (dy2.stride(0) * dy2.element_size()) % 16 != 0:
                dy2 = dy2.contiguous()
            grad_weight = _channel_weight_grad(ctx.sw_ref, partial, ctx.n_channels, dy2, ctx.xkey)
        if ctx.needs_input_grad[0]:
            grad_input = torch.matmul(grad_output, weight)                                      # smt.py:286
        return grad_input, grad_weight, None, None


def _channel_weight_grad(sw_param, partial, n, dy2, xkey):
    """The channel gradient of one module (smt.py:283-284).  Native mode (the parameter owns a GradSink): delivered
    into the padded arena region of the parameter - grouped with the other modules of the backward pass when grouping
    is enabled - and None is returned; otherwise the [n, out_features] gradient is returned.  `xkey` identifies the
    module's input (chunked flushes happen at layer boundaries)."""
    if partial.dtype != dy2.dtype:
        partial = partial.to(dy2.dtype)
    sink = getattr(sw_param, "_smt_sink", None)
    if sink is not None:
        dy2 = _as_operand(dy2)
        accumulate = sink.begin_delivery(sw_param)
        if _grouped["enabled"]:
            _enqueue(xkey, dy2.device, lambda: _pending.add_channel(partial, dy2, n, sink.store, accumulate=accumulate,
                                                                    sq=sink.sq, sq_slot0=sink.sq_slot0, sink=sink))
        else:
            ops.channel_grad_gemm(partial, n, dy2, out=sink.store, accumulate=accumulate)
            sink.sq_ok = False
        return None
    out_f = dy2.shape[1]
    # smt.py:283-284: sum over the batch of partial^T @ dy == ONE contraction over all tokens, on the same tcgen05
    # pipeline as the block gradients (fp32 accumulation, one rounding)
    if n == 0:
        return torch.zeros(0, out_f, dtype=dy2.dtype, device=dy2.device)
    if dy2.dtype == torch.float32 or out_f % 64 != 0:
        return _channel_grad_by_blocks(partial, n, dy2)
    return ops.channel_grad_gemm(partial, n, dy2)


def _channel_grad_by_blocks(partial, n, dy2):
    """fp32 (parity configuration) / odd widths: the same contraction through the single-problem block-gradient entry
    point - every 64 x 64 block of the [n64, out64] result - followed by an un-tiling copy."""
    b = 64
    T, out_f = dy2.shape
    n64 = partial.shape[1]
    if n64 % b:
        partial = torch.nn.functional.pad(partial, (0, b - n64 % b))
        n64 = partial.shape[1]
    out64 = (out_f + b - 1) // b * b
    if out64 != out_f:
        dy2 = torch.nn.functional.pad(dy2, (0, out64 - out_f))
    rows, cols = n64 // b, out64 // b
    rc = ops.make_block_rc([(r, c) for r in range(rows) for c in range(cols)], dy2.device)
    tiles = ops.block_grad_gemm(dy2.contiguous(), partial.contiguous(), rc, b, out_dtype=dy2.dtype)
    full = tiles.view(rows, cols, b, b).permute(0, 2, 1, 3).reshape(n64, out64)
    return full[:n, :out_f].contiguous()


class LinearLayer_ChannelSparsity(nn.Module):
    """Linear layer whose only trainable parameter is a compact copy of its selected input channels (weight columns).
    Reference: smt.py:185-217 (same constructor signature and attribute names; column semantics, see above)."""

    def __init__(self, weight, bias=None, index_list=[]):
        super().__init__()
        if not weight.is_cuda:
            raise SMTLibraryError("LinearLayer_ChannelSparsity needs its weight on a CUDA device: the SMT kernels "
                                  "have no CPU fallback")
        self.weight = weight
        self.weight.requires_grad = False                 # smt.py:191
        self.bias = bias                                  # kept but unused, like smt.py:192,214
        self.index_list = index_list
        seen = set()
        for i in index_list:
            if not 0 <= int(i) < weight.shape[1]:
                raise IndexError(f"channel {i} outside a weight with {weight.shape[1]} input channels")
            if int(i) in seen:
                raise ValueError(f"channel {i} selected twice")
            seen.add(int(i))
        n = len(index_list)
        compact = torch.empty(n, weight.shape[0], dtype=weight.dtype, device=weight.device)
        if n:
            ops.column_gather(weight.data, _channel_idx_for(index_list, weight.device), compact)
        self.selected_weight = nn.Parameter(compact, requires_grad=True)
        self.selected_weight._smt_owner = weakref.ref(self)   # lets SMTAdam find the dense weight to write back
        self.fn = linearChannel.apply
        # Set ONLY by `mark_synced()` (SMTAdam after its fused column write-back); see LinearLayer_MatrixSparsity.
        self._synced = None

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._synced = None
        return out

    # -- what SMTAdam's arena (optim._Arena) asks of the layer that owns a parameter (see LinearLayer_MatrixSparsity) --
    def _arena_ok(self) -> bool:
        """bf16 layers with selected channels and out_features % 64 == 0 take the native path (gradients delivered into
        the arena, fused column write-back); any other channel layer is an ordinary arena parameter, as before."""
        w = self.weight
        return len(self.index_list) > 0 and w.dtype == torch.bfloat16 and self.selected_weight.dtype == w.dtype \
            and w.shape[0] % 64 == 0

    def _grad_tiles(self):
        """(b, row tiles, column tiles) of this layer's channel-gradient launches (ops.channel_grad_gemm)."""
        n, out_f = len(self.index_list), self.weight.shape[0]
        b = ops.channel_grad_block(n, out_f)
        return b, (n + b - 1) // b, out_f // b

    def _arena_layout(self):
        """The last row tile of the gradient launch stores ceil(n/b)*b rows (the rows past n are zero), so the arena
        reserves them: selected_weight and its .grad are the first n rows of the region."""
        b, rows, cols = self._grad_tiles()
        return rows * b * self.weight.shape[0], 2 * rows * cols

    def _writeback(self, off: int):
        w = self.weight.data
        out_f = w.shape[0]
        return ("columns", w.dtype), [(w, int(c), off + i * out_f) for i, c in enumerate(self.index_list)]

    @staticmethod
    def _writeback_args(key, entries, device) -> dict:
        return dict(columns=ops.make_column_table(entries, device), n_columns=len(entries), w_dtype=key[1])

    def mark_synced(self) -> None:
        """Called by SMTAdam right after it has written the updated channels into the columns of `weight` itself; the
        same rule as LinearLayer_MatrixSparsity.mark_synced (storage pointer + version counter of selected_weight)."""
        self._synced = (self.selected_weight.data_ptr(), self.selected_weight._version)

    def sync_weight(self, force: bool = False) -> None:
        """compact -> dense write-back (smt.py:208-211): one launch on every forward, like the reference's loop —
        whatever optimizer updated `selected_weight` (also through `.data` or an aliased flat buffer) is seen.  The only
        exception is right after an SMTAdam step that wrote the columns itself (see `mark_synced`)."""
        if not force and self._synced is not None and \
                self._synced == (self.selected_weight.data_ptr(), self.selected_weight._version):
            return
        self._synced = None
        if len(self.index_list):
            sw = self.selected_weight.data
            if sw.dtype != self.weight.dtype:
                sw = sw.to(self.weight.dtype)
            ops.column_scatter(self.weight.data, _channel_idx_for(self.index_list, self.weight.device),
                               sw.contiguous())

    def forward(self, x):
        self.sync_weight()
        return self.fn(x, self.selected_weight, self.index_list, self.weight)   # smt.py:213


_SPARSE_LAYERS = (LinearLayer_MatrixSparsity, LinearLayer_ChannelSparsity)


def convert_linear_layer_to_channel_sparsity(model,
                                             selected_channel,
                                             selected_channel_attention,
                                             part_module_name=['.layers']):
    """Reference: smt.py:25-80.  MLP Linears are looked up in `selected_channel`, attention Linears (q/k/v/o by
    substring) in `selected_channel_attention`; only weights that still require grad are converted."""
    names = [name for name, module in model.named_modules()
             if isinstance(module, nn.Linear) and any(part in name for part in part_module_name)]
    for name in names:
        for marker, kind_of, table in (("mlp", _mlp_kind, selected_channel),
                                       ("self_attn", _attn_kind, selected_channel_attention)):
            if marker not in name:
                continue
            module = _getattr_path(model, name)
            if not isinstance(module, nn.Linear) or not module.weight.requires_grad:
                continue
            _rank0_print(f"Module Test: {name}")
            index_list = table[(kind_of(name), _layer_of(name))]
            sparse = LinearLayer_ChannelSparsity(module.weight, bias=None, index_list=index_list)
            _setattr_path(model, name, sparse.to(module.weight.device).to(module.weight.dtype))
    return model


def convert_channel_sparsity_to_linear_layer(model, part_module_name=['.layers']):
    """Write the trained channels back and restore plain nn.Linear modules (the channel twin of smt.py:416-457; the
    reference has no such function for channels)."""
    unfuse_qkv_projections(model)
    names = [name for name, module in model.named_modules()
             if isinstance(module, LinearLayer_ChannelSparsity) and any(part in name for part in part_module_name)]
    for name in names:
        module = _getattr_path(model, name)
        module.sync_weight(force=True)
        out_f, in_f = module.weight.shape
        linear = nn.Linear(in_f, out_f, bias=False, device="meta")
        linear = linear.to_empty(device=module.weight.device).to(module.weight.dtype)
        linear.weight = module.weight
        _setattr_path(model, name, linear)
    return model


def freeze_unselected_channel_layer(model,
                                    select_parameters,
                                    select_attention_parameters,
                                    mixture=False):
    """Reference: smt.py:748-831.  Attention names resolve to q/k/v only here (o_proj -> None, smt.py:778,811)."""
    for name, param in model.named_parameters():
        layer = _layer_of(name)
        if "mlp" in name:
            trainable = (_mlp_kind(name), layer) in select_parameters.keys()
        elif "self_attn" in name:
            kind = next((k for k in ("q_proj", "k_proj", "v_proj") if k in name), None)
            table = select_parameters if mixture else select_attention_parameters
            trainable = (kind, layer) in table.keys()
        else:
            trainable = False
        param.requires_grad = trainable
    return model
