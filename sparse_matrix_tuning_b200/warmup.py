"""On-device warm-up score accumulation — replaces the per-step capture loop of the reference driver.

Reference (paths relative to the reference root):
  deepspeed/fine_tune.py:716-768   after every warm-up backward: for each q/k/v (and, if the MLP ratio is > 0,
                                   gate/up/down) weight, `safe_get_full_grad(p).detach().cpu().to(float32)` is
                                   summed into a dict keyed (module_name, layer)  — 1.6 GB (q/k/v) to 11 GB (with
                                   MLP) of blocking D2H per step for LLaMA-3-8B, 3.2-25 GB of CPU state.
  deepspeed/fine_tune.py:649-678   activation hook: |x|, barrier, all_reduce of the full activation, D2H, `+=`.

Here the accumulators live in HBM and are updated by `smt_score_accumulate` (elementwise, any strategy,
10 B/element) or `smt_block_sum_accumulate` (per-block signed sums, 2 B/element, exact for the `mean_abs`
statistic that q/k/v always use — fine_tune.py:306-313 never forwards `calculate_strategy`).  Nothing crosses PCIe.
"""
from __future__ import annotations

import re
import weakref
from typing import Callable, Dict, Iterable, Optional, Tuple

import torch

from . import ops
from ._lib import SMTLibraryError

_LAYER_RE = re.compile(r"model\.layers\.(\d+)\.")
Key = Tuple[str, Optional[int]]


def classify_parameter(name: str, mlp: bool, attention: bool) -> Optional[Key]:
    """(module_name, layer) exactly as fine_tune.py:718-750 derives it, or None if the parameter is not captured."""
    m = _LAYER_RE.search(name)
    layer = int(m.group(1)) if m else None
    if "mlp" in name and mlp:                                           # fine_tune.py:723
        kind = "gate_proj" if "gate_proj" in name else "up_proj" if "up_proj" in name else "down_proj"
        return (kind, layer)
    if "self_attn" in name and "weight" in name and attention:          # fine_tune.py:744
        for kind in ("q_proj", "k_proj", "v_proj"):                     # fine_tune.py:747 (o_proj excluded)
            if kind in name:
                return (kind, layer)
    return None


class WarmupGradAccumulator:
    """Sum over warm-up steps of the (already data-parallel-reduced) gradients of the targeted weights.

    mode="elementwise": fp32 accumulator per matrix (what the reference keeps on the CPU) — works with every
                        calculate_strategy.
    mode="block_sum":   one fp32 signed sum per b x b block — 65 536x smaller, valid for `mean_abs` only.
    """

    def __init__(self, block: int = 256, mode: str = "elementwise", mlp: bool = False, attention: bool = True):
        if mode not in ("elementwise", "block_sum"):
            raise ValueError(mode)
        self.block, self.mode, self.mlp, self.attention = block, mode, mlp, attention
        self.acc: Dict[Key, torch.Tensor] = {}
        self.shapes: Dict[Key, Tuple[int, int]] = {}
        self.steps = 0

    def accumulate(self, named_parameters: Iterable, grad_of: Optional[Callable] = None) -> None:
        """Call once after each warm-up backward. `grad_of(param)` defaults to `param.grad`
        (pass deepspeed's `safe_get_full_grad` under ZeRO)."""
        for name, p in named_parameters:
            key = classify_parameter(name, self.mlp, self.attention)
            if key is None:
                continue
            g = p.grad if grad_of is None else grad_of(p)
            if g is None:
                continue
            self.add(key, g.detach())
        self.steps += 1

    def attach(self, model, free_grads: bool = False):
        """Hook mode (SURVEY.md §8f row 3): accumulate each targeted gradient the moment autograd has finished
        producing it (`register_post_accumulate_grad_hook`) instead of sweeping all parameters after backward.
        With `free_grads=True` the parameter's `.grad` is released right away, so a capture-only warm-up pass never
        holds more than one targeted gradient at a time.  Returns the hook handles (call `.remove()` on each, or
        `detach()`)."""
        self._handles = []
        for name, p in model.named_parameters():
            key = classify_parameter(name, self.mlp, self.attention)
            if key is None or not p.requires_grad:
                continue

            def hook(param, key=key):
                if param.grad is not None:
                    self.add(key, param.grad.detach())
                    if free_grads:
                        param.grad = None

            self._handles.append(p.register_post_accumulate_grad_hook(hook))
        return self._handles

    def detach(self) -> None:
        for h in getattr(self, "_handles", []):
            h.remove()
        self._handles = []

    def add(self, key: Key, grad: torch.Tensor) -> None:
        if not grad.is_cuda:
            raise SMTLibraryError("WarmupGradAccumulator works on CUDA gradients (no CPU path)")
        if grad.dim() != 2:
            raise SMTLibraryError(f"gradient of {key} is not a matrix")
        if grad.stride(1) != 1:
            grad = grad.contiguous()
        R, C = grad.shape
        b = self.block
        if key not in self.acc:
            self.shapes[key] = (R, C)
            shape = (R, C) if self.mode == "elementwise" else (R // b, C // b)
            self.acc[key] = torch.zeros(shape, dtype=torch.float32, device=grad.device)
        if self.mode == "elementwise":
            ops.score_accumulate(self.acc[key], grad.contiguous())
        else:
            ops.block_sum_accumulate(self.acc[key], grad, b)

    # -- hand-off to selection ------------------------------------------------------------------------
    def grads(self) -> Dict[Key, torch.Tensor]:
        """The reference's `attention_warmup_grads` / `warmup_grads` dict, resident in HBM (elementwise mode)."""
        if self.mode != "elementwise":
            raise SMTLibraryError("block_sum mode keeps no full-size gradients; use scores()")
        return dict(self.acc)

    def scores(self, calculate_strategy: str = "mean_abs"):
        """(keys, [R/b, C/b] score tensors) ready for smt_helper.select_submatrix_from_scores."""
        keys = list(self.acc.keys())
        if self.mode == "block_sum":
            if calculate_strategy != "mean_abs":
                raise SMTLibraryError("block_sum accumulation is linear in g and only reproduces 'mean_abs'")
            return keys, [ops.block_sum_finalize(self.acc[k], self.block) for k in keys]
        return keys, [ops.block_score_reduce(self.acc[k], self.block, calculate_strategy) for k in keys]

    def flat_state(self) -> torch.Tensor:
        """All accumulators as one flat tensor (block_sum mode: the tensor a DP job all-reduces per step)."""
        return torch.cat([self.acc[k].reshape(-1) for k in self.acc])

    def load_flat_state(self, flat: torch.Tensor) -> None:
        off = 0
        for k in self.acc:
            n = self.acc[k].numel()
            self.acc[k].copy_(flat[off:off + n].view_as(self.acc[k]))
            off += n


class FactoredBlockSumAccumulator:
    """Block sums of the targeted weight gradients of a FROZEN model, built from activations and output gradients.

    For y = x W^T the signed sum of block (r, c) of dW factors over the tokens t:
        sum_{o in r, k in c} dW[o, k] = sum_t Dy[t, r] * X[t, c],
    Dy[t, r] = sum_{o in r} dy[t, o] and X[t, c] = sum_{k in c} x[t, k].  A forward hook on every targeted nn.Linear
    reduces its input to X (`ops.token_block_sums`, one read of x; x itself is not kept), a tensor hook on its output
    reduces dy to Dy in backward and adds Dy^T X to the module's [R/b, C/b] accumulator (`ops.block_outer_accumulate`).
    No weight gradient is ever formed, so the model stays frozen and the warm-up pass can run the same fused path as
    the training step (`fuse_qkv_projections`, `fuse_causal_lm_loss`).

    Same surface as `WarmupGradAccumulator(mode="block_sum")` - `acc` / `shapes` keyed (module_name, layer),
    `scores("mean_abs")`, `flat_state()` / `load_flat_state()` - so `dp.allreduce_block_sums` and
    `smt_helper.select_submatrix_from_scores` take it unchanged.  Only `mean_abs` is linear in the gradient; `abs_mean`,
    `L1` and `L2` need `WarmupGradAccumulator(mode="elementwise")`.

    Usage - freezing is the caller's job:
        for p in model.parameters(): p.requires_grad_(False)
        model.enable_input_require_grads()          # the hidden states must require grad for dy to exist
        fuse_qkv_projections(model); fuse_causal_lm_loss(model)            # optional
        acc = FactoredBlockSumAccumulator(block=256).attach(model)  ... warm-up passes (forward + backward) ...
        acc.detach(); keys, scores = acc.scores("mean_abs"); sel = select_submatrix_from_scores(keys, scores, n)
        unfuse_qkv_projections(model)
        freeze_unselected_matrix_layer(...); convert_linear_layer_to_matrix_sparsity(...); fuse_qkv_projections(model)
    Forwards whose output does not require grad (`no_grad` evaluation, the first forward of reentrant checkpointing)
    are ignored; the forward that non-reentrant checkpointing recomputes costs one more X pass and adds nothing.
    """

    def __init__(self, block: int = 256, mlp: bool = False, attention: bool = True):
        self.block, self.mlp, self.attention = block, mlp, attention
        self.acc: Dict[Key, torch.Tensor] = {}
        self.shapes: Dict[Key, Tuple[int, int]] = {}
        self._handles = []
        self._x_cache = None         # (weakref to the last input, its version, its X): q/k/v share their input

    def attach(self, model) -> "FactoredBlockSumAccumulator":
        """Forward hooks on q/k/v (and gate/up/down with mlp=True) of `model`; o_proj is never captured
        (fine_tune.py:747).  Accumulators are created here, in module order.  Returns self."""
        b = self.block
        found = []
        for name, mod in model.named_modules():
            if not isinstance(mod, torch.nn.Linear):
                continue
            key = classify_parameter(name + ".weight", self.mlp, self.attention)
            if key is None:
                continue
            R, Cc = mod.weight.shape
            if R % b or Cc % b:
                raise SMTLibraryError(f"{name}: weight {R}x{Cc} is not a multiple of the block size {b}")
            found.append((key, mod, R, Cc))
        for key, mod, R, Cc in found:
            if key not in self.acc:
                self.shapes[key] = (R, Cc)
                self.acc[key] = torch.zeros((R // b, Cc // b), dtype=torch.float32, device=mod.weight.device)
            self._handles.append(mod.register_forward_hook(lambda _m, args, out, key=key: self._forward(key, args[0], out)))
        return self

    def detach(self) -> None:
        for h in self._handles:
            h.remove()
        self._handles = []
        self._x_cache = None

    def _forward(self, key: Key, x: torch.Tensor, out: torch.Tensor) -> None:
        if not (torch.is_grad_enabled() and out.requires_grad):
            return
        if not (x.is_cuda and out.is_cuda):
            raise SMTLibraryError("FactoredBlockSumAccumulator works on CUDA activations (no CPU path)")
        c = self._x_cache
        if c is not None and c[0]() is x and c[1] == x._version:
            X = c[2]
        else:
            X = ops.token_block_sums(_rows(x), self.block)
            self._x_cache = (weakref.ref(x), x._version, X)
        acc = self.acc[key]
        out.register_hook(lambda dy: ops.block_outer_accumulate(acc, ops.token_block_sums(_rows(dy), self.block), X))

    def scores(self, calculate_strategy: str = "mean_abs"):
        """(keys, [R/b, C/b] score tensors) ready for smt_helper.select_submatrix_from_scores."""
        if calculate_strategy != "mean_abs":
            raise SMTLibraryError("factored block sums are linear in the gradient and only reproduce 'mean_abs'")
        keys = list(self.acc.keys())
        return keys, [ops.block_sum_finalize(self.acc[k], self.block) for k in keys]

    flat_state = WarmupGradAccumulator.flat_state
    load_flat_state = WarmupGradAccumulator.load_flat_state


def _rows(t: torch.Tensor) -> torch.Tensor:
    """[..., F] -> [T, F] with unit column stride and a 16-byte aligned base and row pitch."""
    t2 = t.reshape(-1, t.shape[-1])
    if t2.stride(1) != 1 or t2.data_ptr() % 16 or (t2.stride(0) * t2.element_size()) % 16:
        t2 = t2.clone(memory_format=torch.contiguous_format)
    return t2


class WarmupActivationAccumulator:
    """sum over warm-up steps of sum_b |x[b, S, C]| per Linear input — the part of the activation hook
    (fine_tune.py:649-678) that select_channel_based_on_activation actually consumes (smt_helper.py:170)."""

    def __init__(self):
        self.acc: Dict[Key, torch.Tensor] = {}

    def add(self, key: Key, x: torch.Tensor) -> None:
        if not x.is_cuda:
            raise SMTLibraryError("WarmupActivationAccumulator works on CUDA activations (no CPU path)")
        if x.dim() == 2:
            x = x.unsqueeze(0)
        x = x.detach().contiguous()
        if key not in self.acc:
            self.acc[key] = torch.zeros(x.shape[1:], dtype=torch.float32, device=x.device)
        ops.act_score_accumulate(self.acc[key], x)

    def attach(self, model, mlp: bool = True, attention: bool = True):
        """Forward pre-hooks on every targeted nn.Linear of `model` (all of a decoder's Linears in the reference,
        fine_tune.py:680-689): accumulates sum_b |x| of each module's INPUT.  Keys are (module_name, layer) as in
        fine_tune.py:659-677 (o_proj is captured too, like the reference's hook)."""
        self._handles = []
        for name, mod in model.named_modules():
            if not isinstance(mod, torch.nn.Linear):
                continue
            m = _LAYER_RE.search(name + ".")
            layer = int(m.group(1)) if m else None
            key = None
            if "mlp" in name and mlp:
                key = ("gate_proj" if "gate_proj" in name else "up_proj" if "up_proj" in name else "down_proj", layer)
            elif "self_attn" in name and attention:
                for kind in ("q_proj", "k_proj", "v_proj", "o_proj"):
                    if kind in name:
                        key = (kind, layer)
            if key is None:
                continue
            self._handles.append(mod.register_forward_pre_hook(lambda _m, args, key=key: self.add(key, args[0])))
        return self._handles

    def detach(self) -> None:
        for h in getattr(self, "_handles", []):
            h.remove()
        self._handles = []

    def activations(self) -> Dict[Key, torch.Tensor]:
        return dict(self.acc)
