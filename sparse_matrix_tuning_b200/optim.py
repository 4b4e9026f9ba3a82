"""`SMTAdam`: the compact AdamW step of the SMT phase as ONE fused sm_100a kernel per parameter group.

Reference call sites replaced (paths relative to the reference root):
  deepspeed/fine_tune.py:352-363   `FusedAdam(optimizer_grouped_parameters, lr=ft_learning_rate, betas=(0.9, 0.95))`
  deepspeed/fine_tune.py:379-384   `deepspeed.initialize(... optimizer=new_optimizer ...)` — bf16 params with fp32
                                   masters and `gradient_clipping: 1.0` (helpers/deepspeed_helpers.py:87)
  deepspeed/fine_tune.py:773       `model.step()`
  deepspeed/smt/smt.py:332-341     the per-forward scatter of the updated blocks into the dense weight

The constructor accepts FusedAdam's keyword arguments, so the driver line at fine_tune.py:352 works unchanged
with `AdamOptimizer = SMTAdam`.  It is a regular `torch.optim.Optimizer` (param_groups, state_dict, LR
schedulers work).

Memory layout (`flatten=True`, the default): each parameter group becomes one flat arena — `flat_param` and
`flat_grad` in the parameter dtype, fp32 `master` / `exp_avg` / `exp_avg_sq` — and every parameter's `.data`
and `.grad` are re-pointed to views of it.  `flat_grad` is therefore the single buffer a data-parallel step
all-reduces (see dp.py), and `linearZ.backward` writes block gradients straight into it.  One `smt_grad_sqnorm`
+ one `smt_compact_adam` launch per group then performs: optional 1/world scaling, global-norm clip, AdamW on the
fp32 masters, rounding to the parameter dtype into `flat_param`, and the write-back of every updated block into
its dense weight matrix.

Gradient delivery protocol (`GradSink`).  Every `selected_weight` of an arena owns a `GradSink`: the view of
`flat_grad` that `linearZ.backward` writes into, plus three host-side flags.  bf16 channel layers
(`LinearLayer_ChannelSparsity`) take part the same way: `linearChannel.backward` delivers into the arena, whose region for
such a parameter has the padding rows of the gradient launch's last row tile, and one `smt_compact_adam_columns` launch
writes the updated channels into their weight columns.  `zero_grad()` is LAZY for those
parameters: it only sets `sink.overwrite`, and the first block-gradient GEMM that delivers afterwards overwrites the
view instead of accumulating (per-work-item flag) - the 114 MB memset and the read-modify-write of the GEMM epilogue
disappear from the step.  Further backward passes before the next `step()` accumulate (gradient accumulation).  The
same epilogue emits the sum of squares of every block it stores (`block_sq`), so the clip norm needs no pass over the
buffer either; whenever those partial sums cannot be trusted (split-K launches, an all-reduce touched the buffer, a
gradient was copied in from elsewhere) `step()` falls back to `smt_grad_sqnorm`.  Parameters whose `.grad` was
dropped or replaced behind the optimizer's back (`model.zero_grad()` sets it to None) are handled: the sink re-attaches
itself at the next backward and starts from an overwrite; parameters without a sink are copied into the arena.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import ops
from ._lib import SMTLibraryError


def _owner_of(p):
    """The SMT layer whose dense weight SMTAdam writes `p` back into, or None.  An owner provides (smt/smt.py):
    `_arena_layout()` -> (elements the arena reserves, sum-of-squares slots), `_writeback(offset)` -> (key, table
    entries), `_writeback_args(key, entries, device)` -> ops.compact_adam keyword arguments, `mark_synced()` and
    `sync_weight(force)`."""
    ref = getattr(p, "_smt_owner", None)
    owner = ref() if ref is not None else None
    return owner if owner is not None and owner._arena_ok() else None


def _writeback_args(owners_offs, device):
    """ops.compact_adam keyword arguments of ONE launch that writes back the parameters [(owner, arena offset)], or
    None when they need different kinds of table (blocks of another size or dtype, columns)."""
    key, entries = None, []
    for owner, off in owners_offs:
        k, e = owner._writeback(off)
        if key is not None and k != key:
            return None
        key = k
        entries += e
    return type(owners_offs[0][0])._writeback_args(key, entries, device)


def _cached_writeback_args(cache: dict, slot, owners_offs, device):
    """`_writeback_args`, rebuilt only when a dense weight's storage moved."""
    wkey = tuple((o.weight.data_ptr(), o.weight.stride(0)) for o, _ in owners_offs)
    hit = cache.get(slot)
    if hit is None or hit[0] != wkey:
        hit = (wkey, _writeback_args(owners_offs, device))
        cache[slot] = hit
    return hit[1]


class GradSink:
    """Where `linearZ.backward` / `linearChannel.backward` deliver the gradient of one `selected_weight` in native
    mode."""
    __slots__ = ("view", "store", "sq", "sq_slot0", "overwrite", "touched", "sq_ok", "__weakref__")

    def __init__(self, view: torch.Tensor, sq: Optional[torch.Tensor], sq_slot0: int, store: Optional[torch.Tensor] = None):
        self.view = view              # the parameter's .grad: a view of the arena's flat_grad
        self.store = view if store is None else store   # what the GEMM writes: `view` plus the padding rows of a
                                                        # channel parameter ([ceil(n/b)*b, out_features])
        self.sq = sq                  # the arena's per-tile sum-of-squares slots (2 per block / channel tile) or None
        self.sq_slot0 = sq_slot0
        self.overwrite = False        # the next delivery replaces the contents (lazy zero_grad)
        self.touched = False          # a gradient was delivered since the last zero_grad
        self.sq_ok = False            # the slots hold the sum of squares of what the view stores now

    def begin_delivery(self, param) -> bool:
        """Called by linearZ.backward before it writes.  Returns True when the delivery must ACCUMULATE."""
        g = param.grad
        if g is None or g.data_ptr() != self.view.data_ptr():
            # somebody dropped / replaced .grad (model.zero_grad(set_to_none=True), `p.grad = None`): whatever the
            # arena still holds is stale - start over and re-attach the view
            self.overwrite = True
            param.grad = self.view
        accumulate = not self.overwrite
        self.overwrite = False
        self.touched = True
        return accumulate


class _Arena:
    """Flat storage of one parameter group."""

    def __init__(self, params: List[torch.nn.Parameter]):
        first = params[0]
        self.params = params
        self.device = first.device
        self.dtype = first.dtype
        offs, sizes, slots, total = [], [], [], 0
        for p in params:
            if p.device != self.device or p.dtype != self.dtype:
                raise SMTLibraryError("SMTAdam: all parameters of a group must share device and dtype")
            owner = _owner_of(p)
            size, n_sq = owner._arena_layout() if owner is not None else (p.numel(), 0)
            offs.append(total)
            sizes.append((size + 7) // 8 * 8)               # kernels work on 8-element vectors
            slots.append(n_sq)
            total += sizes[-1]
        self.offsets, self.sizes, self.sq_counts, self.total = offs, sizes, slots, total
        self.flat_param = torch.zeros(total, dtype=self.dtype, device=self.device)
        self.flat_grad = torch.zeros(total, dtype=self.dtype, device=self.device)
        self.master = torch.zeros(total, dtype=torch.float32, device=self.device)
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=self.device)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=self.device)
        self.sqnorm = torch.zeros(1, dtype=torch.float32, device=self.device)
        # two sum-of-squares slots per selected block / channel tile (written by the gradient GEMM epilogue)
        self.block_sq = torch.zeros(max(sum(slots), 1), dtype=torch.float32, device=self.device)
        self.sq_dirty = True                                # the buffer was modified by something else (all-reduce, copy)
        self.sq_override: Optional[torch.Tensor] = None     # partial sums supplied by a data-parallel exchange
        self.sinks: List[Optional[GradSink]] = []
        self.grad_views: List[torch.Tensor] = []
        slot = 0
        for p, off, size, n_sq in zip(params, offs, sizes, slots):
            n = p.numel()
            view = self.flat_param[off:off + n].view(p.shape)
            view.copy_(p.data)
            self.master[off:off + n].copy_(p.data.reshape(-1).float())
            p.data = view
            g = self.flat_grad[off:off + n].view(p.shape)
            if p.grad is not None:
                g.copy_(p.grad)
            p.grad = g
            self.grad_views.append(g)
            if _owner_of(p) is not None:
                store = self.flat_grad[off:off + size].view(-1, *p.shape[1:]) if size != n else g
                sink = GradSink(g, self.block_sq, slot, store)
                slot += n_sq
                p._smt_sink = sink                          # linearZ / linearChannel.backward deliver here directly
                self.sinks.append(sink)
            else:
                self.sinks.append(None)
        self.all_sinks = all(sk is not None for sk in self.sinks)
        self._writeback_cache: dict = {}

    def reconcile_grads(self) -> None:
        """Before a step: every parameter's gradient must be what the arena holds.
        * sink parameters that received nothing since zero_grad(): their slice (and slots) become zero;
        * parameters without a sink (e.g. layer norms in mixture mode) whose `.grad` is no longer the arena view
          (autograd created a fresh tensor after `set_to_none`): copied in and re-attached; None -> zeros."""
        for p, view, sink, n_slots in zip(self.params, self.grad_views, self.sinks, self.sq_counts):
            if sink is not None:
                if p.grad is None or p.grad.data_ptr() != view.data_ptr():
                    if not sink.touched:                    # dropped and never delivered again: no gradient this step
                        sink.overwrite = True
                    p.grad = view
                if sink.overwrite:                          # nothing was delivered since the (lazy) zero_grad
                    view.zero_()                            # (padding rows of a channel parameter only ever hold zeros)
                    self.block_sq[sink.sq_slot0:sink.sq_slot0 + n_slots].zero_()
                    sink.overwrite = False
                    sink.sq_ok = True
            else:
                g = p.grad
                if g is None:
                    view.zero_()
                    self.sq_dirty = True
                elif g.data_ptr() != view.data_ptr():
                    view.copy_(g)
                    self.sq_dirty = True
                p.grad = view

    def sq_partials(self) -> Optional[torch.Tensor]:
        """Partial sums of squares that add up to |flat_grad|^2, or None when a full pass is needed."""
        if self.sq_override is not None:
            return self.sq_override
        if self.sq_dirty or not self.all_sinks or not all(sk.sq_ok for sk in self.sinks):
            return None
        return self.block_sq

    def fused_writeback(self):
        """ops.compact_adam write-back arguments of ONE launch over the whole arena, or None when the group is not
        purely SMT parameters with one kind of table (blocks of one size and weight dtype, or channels of one weight
        dtype); the step then falls back to per-parameter launches."""
        owners = [_owner_of(p) for p in self.params]
        if any(o is None for o in owners):
            return None
        return _cached_writeback_args(self._writeback_cache, "all", list(zip(owners, self.offsets)), self.device)

    def writeback(self, i: int):
        """ops.compact_adam write-back arguments of parameter i alone (offsets relative to its slice), or None."""
        owner = _owner_of(self.params[i])
        if owner is None:
            return None
        return _cached_writeback_args(self._writeback_cache, i, [(owner, 0)], self.device)


class SMTAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, bias_correction=True, betas=(0.9, 0.999), eps=1e-8, adam_w_mode=True,
                 weight_decay=0.0, amsgrad=False, set_grad_none=False, max_grad_norm=0.0, flatten=True,
                 grad_scale=1.0):
        if amsgrad:
            raise SMTLibraryError("SMTAdam: amsgrad is not supported (neither does FusedAdam)")
        if not adam_w_mode or not bias_correction:
            raise SMTLibraryError("SMTAdam implements FusedAdam's default adam_w_mode with bias correction only")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        super().__init__(params, defaults)
        self.max_grad_norm = float(max_grad_norm)
        self.grad_scale = float(grad_scale)                # e.g. 1/world_size after a SUM all-reduce
        self.steps_done = 0                                # serial number of the gradient state (bumped by every step())
        self.flatten = bool(flatten)
        self._loose_writeback: dict = {}                   # flatten=False: write-back tables per parameter
        self._arenas: List[Optional[_Arena]] = []
        for group in self.param_groups:
            group.setdefault("step", 0)
            ps = [p for p in group["params"] if p.requires_grad]
            for p in ps:
                if not p.is_cuda:
                    raise SMTLibraryError("SMTAdam: parameters must live on a CUDA device (no CPU fallback)")
            self._arenas.append(_Arena(ps) if (self.flatten and ps) else None)
        self._publish_state()

    # -- introspection ---------------------------------------------------------------------------------
    def flat_grads(self) -> List[torch.Tensor]:
        """The flat gradient buffers (one per non-empty group) — what a data-parallel step all-reduces."""
        return [a.flat_grad for a in self._arenas if a is not None]

    def snapshot(self) -> dict:
        """Deep copy of everything a step changes (flat parameters, fp32 masters and moments, step counters) - lets a
        harness try a step and take it back (bench.py's data-parallel check)."""
        snap = {"steps": [g["step"] for g in self.param_groups], "arenas": [], "grad_scale": self.grad_scale}
        for arena in self._arenas:
            snap["arenas"].append(None if arena is None else
                                  tuple(t.clone() for t in (arena.flat_param, arena.master, arena.exp_avg, arena.exp_avg_sq)))
        return snap

    @torch.no_grad()
    def restore(self, snap: dict) -> None:
        self.grad_scale = snap["grad_scale"]
        for g, st in zip(self.param_groups, snap["steps"]):
            g["step"] = st
        for arena, saved in zip(self._arenas, snap["arenas"]):
            if arena is None:
                continue
            for dst, src in zip((arena.flat_param, arena.master, arena.exp_avg, arena.exp_avg_sq), saved):
                dst.copy_(src)
            for p in arena.params:
                owner = _owner_of(p)
                if owner is not None:
                    owner.sync_weight(force=True)            # dense blocks <- restored compact values
                    owner.mark_synced()

    def trainable_elements(self) -> int:
        return sum(p.numel() for g in self.param_groups for p in g["params"] if p.requires_grad)

    def _publish_state(self) -> None:
        # expose per-parameter views so torch's state_dict()/schedulers see ordinary Adam state
        for group, arena in zip(self.param_groups, self._arenas):
            if arena is None:
                continue
            for p, off in zip(arena.params, arena.offsets):
                n = p.numel()
                self.state[p] = {"exp_avg": arena.exp_avg[off:off + n].view(p.shape),
                                 "exp_avg_sq": arena.exp_avg_sq[off:off + n].view(p.shape),
                                 "master": arena.master[off:off + n].view(p.shape)}

    def load_state_dict(self, state_dict):
        """Restores hyper-parameters and state IN PLACE.  torch's generic implementation would cast every state tensor
        to the parameter dtype (bf16) and replace the arena views by fresh tensors; the fp32 masters and moments must
        keep their precision and their storage."""
        saved_groups, saved_state = state_dict["param_groups"], state_dict["state"]
        if len(saved_groups) != len(self.param_groups):
            raise ValueError("loaded state dict has a different number of parameter groups")
        id_map = {}
        for sg, g in zip(saved_groups, self.param_groups):
            if len(sg["params"]) != len(g["params"]):
                raise ValueError("loaded state dict contains a parameter group that doesn't match the size of optimizer's group")
            for pid, p in zip(sg["params"], g["params"]):
                id_map[pid] = p
            for k, v in sg.items():
                if k != "params":
                    g[k] = v
        for pid, st in saved_state.items():
            p = id_map[pid]
            mine = self.state[p]
            for name, val in st.items():
                if torch.is_tensor(val):
                    if name in mine and torch.is_tensor(mine[name]):
                        mine[name].copy_(val.reshape(mine[name].shape))       # into the arena view, fp32 preserved
                    else:
                        mine[name] = val.detach().clone().to(p.device)
                else:
                    mine[name] = val

    def zero_grad(self, set_to_none: bool = False):
        """Arena groups: `.grad` views stay attached (nothing is re-pointed).  Parameters fed by `linearZ.backward`
        are zeroed LAZILY - the next block-gradient launch overwrites them (see the module docstring) - the others
        are zeroed in place.  Non-arena groups behave like torch's zero_grad."""
        for group, arena in zip(self.param_groups, self._arenas):
            if arena is not None:
                arena.sq_override = None
                arena.sq_dirty = not arena.all_sinks
                for p, view, sink in zip(arena.params, arena.grad_views, arena.sinks):
                    if sink is not None:
                        sink.overwrite, sink.touched, sink.sq_ok = True, False, False
                    else:
                        view.zero_()
                    p.grad = view
            else:
                for p in group["params"]:
                    if p.grad is not None:
                        if set_to_none:
                            p.grad = None
                        else:
                            p.grad.zero_()

    def mark_grads_modified(self) -> None:
        """Tell the optimizer that something outside the block-gradient GEMM changed the flat gradient buffers (an
        all-reduce, a manual edit): the per-block sums of squares are then stale and the clip norm is recomputed."""
        for arena in self._arenas:
            if arena is not None:
                arena.sq_dirty = True

    # -- the step --------------------------------------------------------------------------------------
    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        from .smt.smt import flush_block_grads
        flush_block_grads()                                  # guard: pending grouped block-gradient launches
        for arena in self._arenas:
            if arena is not None:
                arena.reconcile_grads()
        clip = self.max_grad_norm > 0.0
        total_sq = None
        self.sqnorm_source = None
        if clip:
            live = [a for a in self._arenas if a is not None]
            loose = any(a is None and any(p.grad is not None for p in g["params"])
                        for g, a in zip(self.param_groups, self._arenas))
            partials = live[0].sq_partials() if (len(live) == 1 and not loose) else None
            if partials is not None:
                # sums of squares emitted by the GEMM epilogue (or by the data-parallel exchange): no extra pass
                total_sq = partials
                self.sqnorm_source = "partials"
            else:
                parts = []
                for group, arena in zip(self.param_groups, self._arenas):
                    if arena is not None:
                        parts.append(ops.grad_sqnorm(arena.flat_grad, arena.sqnorm))
                    else:
                        parts += [ops.grad_sqnorm(p.grad.contiguous()) for p in group["params"] if p.grad is not None]
                if len(parts) == 1:
                    total_sq = parts[0]
                elif parts:
                    total_sq = torch.stack([t.reshape(()) for t in parts]).sum().reshape(1)
                self.sqnorm_source = "grad_sqnorm"
        self.last_sqnorm = total_sq                          # tensor(s) the clip used (tests / reports)
        for group, arena in zip(self.param_groups, self._arenas):
            group["step"] += 1
            b1, b2 = group["betas"]
            common = dict(lr=float(group["lr"]), beta1=float(b1), beta2=float(b2), eps=float(group["eps"]),
                          weight_decay=float(group["weight_decay"]), step=int(group["step"]),
                          grad_scale=self.grad_scale, sqnorm=total_sq, max_norm=self.max_grad_norm if clip else 0.0)
            if arena is not None:
                self._step_arena(arena, common)
            else:
                for p in group["params"]:
                    if p.grad is not None:
                        self._step_loose(p, common)
        self.steps_done += 1
        for arena in self._arenas:
            if arena is not None:                            # the step consumed this gradient state
                arena.sq_override = None
                arena.sq_dirty = True
                for sink in arena.sinks:
                    if sink is not None:
                        sink.touched = False
        return loss

    def _step_arena(self, arena: _Arena, common) -> None:
        fused = arena.fused_writeback()
        if fused is not None:
            ops.compact_adam(arena.master, arena.exp_avg, arena.exp_avg_sq, arena.flat_grad,
                             compact_out=arena.flat_param, **fused, **common)
            for p in arena.params:
                _owner_of(p).mark_synced()
            return
        for i, (p, off, n) in enumerate(zip(arena.params, arena.offsets, arena.sizes)):
            sl = slice(off, off + n)
            wb = arena.writeback(i)
            ops.compact_adam(arena.master[sl], arena.exp_avg[sl], arena.exp_avg_sq[sl], arena.flat_grad[sl],
                             compact_out=arena.flat_param[sl], **(wb or {}), **common)
            if wb is not None:
                _owner_of(p).mark_synced()
            else:
                torch.autograd.graph.increment_version(p)   # forward() must re-scatter / autograd must notice

    def _step_loose(self, p, common) -> None:
        """Unflattened mode (e.g. under a wrapper that owns the flat buffers itself): per-parameter state."""
        st = self.state[p]
        n = p.numel()
        if n % 8 != 0 or not p.data.is_contiguous():
            raise SMTLibraryError("SMTAdam(flatten=False): parameters must be contiguous with numel % 8 == 0")
        if "exp_avg" not in st:
            st["exp_avg"] = torch.zeros(n, dtype=torch.float32, device=p.device)
            st["exp_avg_sq"] = torch.zeros(n, dtype=torch.float32, device=p.device)
        if p.dtype == torch.float32:
            master = p.data.reshape(-1)                      # fp32 parameters are their own master
        else:
            if "master" not in st:
                st["master"] = p.data.reshape(-1).float()
            master = st["master"]
        g = p.grad.contiguous().reshape(-1)
        out = None if p.dtype == torch.float32 else p.data.reshape(-1)
        owner = _owner_of(p)
        kw = dict(common)
        if owner is not None:
            kw.update(_cached_writeback_args(self._loose_writeback, id(p), [(owner, 0)], p.device))
        ops.compact_adam(master, st["exp_avg"].reshape(-1), st["exp_avg_sq"].reshape(-1), g, compact_out=out, **kw)
        if owner is not None:
            owner.mark_synced()
        else:
            torch.autograd.graph.increment_version(p)

