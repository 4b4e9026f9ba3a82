"""Merged-weight export and resumable SMT state (SURVEY.md §8f row 1).

The reference saves `model.state_dict()` as is (helpers/deepspeed_helpers.py:341-364): the checkpoint then holds
BOTH `...q_proj.weight` and `...q_proj.selected_weight`, the dense weight lags the compact copy by one optimizer
step (the write-back only happens inside `forward`, smt.py:332-341) and `convert_matrix_sparsity_to_linear_layer`
(smt.py:416-457) is never called by the driver; nothing needed to resume (index lists, optimizer state) is stored.

Here:
  * `merged_state_dict(model)` returns a plain HF-format state dict (no `selected_weight` keys) whose dense weights
    already contain the trained blocks — loadable into an unmodified `LlamaForCausalLM`;
  * `smt_state(model, optimizer)` / `load_smt_state(...)` round-trip what a resume needs: block size, the ordered
    index list of every converted module (the order defines the row layout of `selected_weight`), and the
    optimizer state (fp32 masters, moments, step counters).
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, Optional

import torch

from .smt import smt as _smt


def sparse_modules(model) -> "OrderedDict[str, torch.nn.Module]":
    """Every converted module (block- or channel-sparse), by qualified name."""
    return OrderedDict((n, m) for n, m in model.named_modules() if isinstance(m, _smt._SparseLinear))


def _plain_index(entry):
    """(row, col) block index -> tuple of ints; channel index -> int."""
    return tuple(map(int, entry)) if isinstance(entry, (tuple, list)) else int(entry)


def merged_state_dict(model) -> "OrderedDict[str, torch.Tensor]":
    """State dict of the equivalent dense model: every selected block written back, compact copies dropped."""
    for mod in sparse_modules(model).values():
        mod.sync_weight(force=True)          # one scatter launch per module (no-op cost if SMTAdam already wrote them)
    out = OrderedDict()
    for key, value in model.state_dict().items():
        if key.endswith(".selected_weight"):
            continue
        out[key] = value
    return out


def smt_state(model, optimizer: Optional[torch.optim.Optimizer] = None) -> Dict:
    mods = sparse_modules(model)
    state = {"format": 1,
             "block": {n: getattr(m, "block", None) for n, m in mods.items()},      # None = channel-sparse module
             "index_lists": {n: [_plain_index(e) for e in m.index_list] for n, m in mods.items()},
             "selected_weight": {n: m.selected_weight.detach().clone() for n, m in mods.items()}}
    if optimizer is not None:
        state["optimizer"] = optimizer.state_dict()
    return state


def selection_from_state(state: Dict):
    """Rebuild the two selection dicts `convert_linear_layer_to_matrix_sparsity` takes from saved module names."""
    sel_mlp, sel_attn = {}, {}
    for name, idx in state["index_lists"].items():
        layer = _smt._layer_of(name + ".")
        if "mlp" in name:
            sel_mlp[(_smt._mlp_kind(name), layer)] = list(idx)
        elif "self_attn" in name:
            sel_attn[(_smt._attn_kind(name), layer)] = list(idx)
    return sel_mlp, sel_attn


def load_smt_state(model, state: Dict, optimizer: Optional[torch.optim.Optimizer] = None) -> None:
    """Restore compact parameters (and optimizer state) into an already converted model with the same selection."""
    mods = sparse_modules(model)
    if set(mods) != set(state["index_lists"]):
        raise ValueError("converted modules do not match the checkpoint: "
                         f"{sorted(set(mods) ^ set(state['index_lists']))}")
    for name, mod in mods.items():
        if [_plain_index(e) for e in mod.index_list] != [_plain_index(e) for e in state["index_lists"][name]]:
            raise ValueError(f"index list of {name} differs from the checkpoint (order defines the row layout)")
        with torch.no_grad():
            mod.selected_weight.copy_(state["selected_weight"][name].to(mod.selected_weight.device))
        mod.sync_weight(force=True)
    if optimizer is not None and "optimizer" in state:
        optimizer.load_state_dict(state["optimizer"])       # fp32 masters, moments and step counters, in place
