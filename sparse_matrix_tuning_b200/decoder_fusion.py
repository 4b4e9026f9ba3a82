"""Native kernels for the elementwise work of transformers' LLaMA, Mistral and Qwen3 decoder layers.

Around its GEMMs and attention, an HF `LlamaDecoderLayer` spends most of a training step in short PyTorch ops: the
fp32 round trip of `LlamaRMSNorm` (six passes where one read and one write do), `rotate_half` + cat + three muls and an
add per RoPE tensor, `silu(gate) * up`, and the residual adds; with activation checkpointing all of it runs twice.
`install_layer(layer)` replaces them with the kernels of `csrc/decoder_kernels.cu` through instance-level `forward`
overrides on the layer, its attention, MLP and two norms (`install_norm` for a model's final norm).  Mistral and Qwen3
layers have the same bodies except for the attention (`_FAMILIES`), so one set of overrides serves all three:

  * LlamaRMSNorm       -> one kernel forward (saves fp32 rstd), one backward (dx only: the weight must be frozen);
  * LlamaAttention     -> the HF body with `apply_rotary_pos_emb` replaced by one launch for q and k; Mistral's and
                          Qwen3's bodies also pass `sliding_window` to the attention interface, and Qwen3's per-head
                          `q_norm` / `k_norm` run inside the same launch as RoPE (`QKNormRoPEFn`);
  * LlamaMLP           -> `down_proj(swiglu(gate_proj(x), up_proj(x)))`, projections still called as modules, so SMT
                          modules, the fused q/k/v group and the warm-up hooks see exactly the calls they saw before;
  * LlamaDecoderLayer  -> the residual add after attention runs inside the post-attention norm kernel, and that norm's
                          backward adds the residual stream's gradient in the same pass.

Each override takes the native path only for CUDA bf16 tensors of a supported shape, a frozen norm weight and no KV
cache; anything else runs the class's own `forward`.  The overrides are bound with `types.MethodType`, so
`copy.deepcopy` of a model rebinds them to the copy.  Installed and removed by `smt.fuse_qkv_projections` /
`smt.unfuse_qkv_projections`.

`install_causal_lm(model)` (`smt.fuse_causal_lm_loss`) overrides `<Llama|Mistral|Qwen3>ForCausalLM.forward` so that a
training call with labels runs the frozen lm_head and the causal-LM cross-entropy chunk by chunk
(`LinearCrossEntropyFn`, the kernel of `csrc/loss_kernels.cu`) and never materialises the fp32 logits; such a call
returns `logits=None`.
"""
from __future__ import annotations

import inspect
import threading
import types

import torch
from torch import nn

from . import ops

# ---- install / remove instance-level forward overrides ---------------------------------------------------------------

_OVERRIDE_FLAG = "_smt_forward_override"


def install_forward(module: nn.Module, fn) -> None:
    """`module.forward = fn` bound to `module` (as a method, so that `copy.deepcopy` rebinds it to the copy)."""
    module.forward = types.MethodType(fn, module)
    module.__dict__[_OVERRIDE_FLAG] = True


def remove_forward(module: nn.Module) -> bool:
    """Undo `install_forward`; False when the module had no override."""
    if not module.__dict__.pop(_OVERRIDE_FLAG, False):
        return False
    module.__dict__.pop("forward", None)
    return True


# ---- autograd functions --------------------------------------------------------------------------------------------

class RMSNormFn(torch.autograd.Function):
    """y = rmsnorm(x) * w for a frozen weight."""

    @staticmethod
    def forward(ctx, x, weight, eps):
        y, rstd, _ = ops.rmsnorm_forward(x, weight, eps)
        ctx.save_for_backward(x, weight, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, rstd = ctx.saved_tensors
        dx = ops.rmsnorm_backward(x, weight, rstd, dy.contiguous()) if ctx.needs_input_grad[0] else None
        return dx, None, None


class AddRMSNormFn(torch.autograd.Function):
    """h = res + a, y = rmsnorm(h) * w (frozen weight); returns (h, y).  Backward: dh_total = norm_bwd(dy) + dh."""

    @staticmethod
    def forward(ctx, res, a, weight, eps):
        y, rstd, h = ops.rmsnorm_forward(a, weight, eps, res=res)
        ctx.save_for_backward(h, weight, rstd)
        return h, y

    @staticmethod
    def backward(ctx, dh, dy):
        h, weight, rstd = ctx.saved_tensors
        dx = ops.rmsnorm_backward(h, weight, rstd, dy.contiguous(), dres=dh.contiguous())
        return dx, dx, None, None


class RoPEFn(torch.autograd.Function):
    """(q, k) [B, S, H, 128] -> rotated (q, k), same layout."""

    @staticmethod
    def forward(ctx, q, k, cos, sin):
        ctx.save_for_backward(cos, sin)
        return ops.rope_forward(q, k, cos, sin)

    @staticmethod
    def backward(ctx, dq, dk):
        cos, sin = ctx.saved_tensors
        dq, dk = ops.rope_backward(dq.contiguous(), dk.contiguous(), cos, sin)
        return dq, dk, None, None


class QKNormRoPEFn(torch.autograd.Function):
    """(q, k) [B, S, H, 128] -> per-head RMSNorm (frozen weights wq / wk) then RoPE, same layout (Qwen3 attention)."""

    @staticmethod
    def forward(ctx, q, k, wq, wk, eps_q, eps_k, cos, sin):
        q_out, k_out, rstd_q, rstd_k = ops.qk_norm_rope_forward(q, k, wq, wk, eps_q, eps_k, cos, sin)
        ctx.save_for_backward(q, k, rstd_q, rstd_k, wq, wk, cos, sin)
        return q_out, k_out

    @staticmethod
    def backward(ctx, dq, dk):
        q, k, rstd_q, rstd_k, wq, wk, cos, sin = ctx.saved_tensors
        dq, dk = ops.qk_norm_rope_backward(q, k, wq, wk, rstd_q, rstd_k, cos, sin, dq.contiguous(), dk.contiguous())
        return dq, dk, None, None, None, None, None, None


class SwiGLUFn(torch.autograd.Function):
    """h = silu(g) * u."""

    @staticmethod
    def forward(ctx, g, u):
        ctx.save_for_backward(g, u)
        return ops.swiglu_forward(g, u)

    @staticmethod
    def backward(ctx, dh):
        g, u = ctx.saved_tensors
        dg, du = ops.swiglu_backward(g, u, dh.contiguous())
        return dg, du


# Rows of logits per chunk of `LinearCrossEntropyFn`, a multiple of 256 (the GEMM's M tile, so that results do not depend
# on it).  Measured on one B200 (1 000 W), lm_head + loss forward + backward at T = 8 192, K = 4 096, V = 128 256
# (profiles/r04_causal_lm_loss.md): chunks of 2 048 / 4 096 / 8 192 rows take 14.1-14.4 ms in two runs (medians; single
# repetitions differ by up to 1 ms), with 0.66 / 1.19 / 2.24 GB of peak memory above the inputs; 1 024 rows take
# 14.5-14.7 ms (the input-gradient GEMM then has 64 tiles for 74 CTA pairs).  2 048 is the smallest transient at no
# measured cost.
_CE_CHUNK_ROWS = 2048
_LM_HEAD_TILE_N = 256       # N tile of the fused forward GEMM (smt_fused_linear_forward takes N % 256 == 0)


class LinearCrossEntropyFn(torch.autograd.Function):
    """loss = sum_t CE(h_t W^T, y_t) / denom for h [T, K] (bf16) and a frozen W [V, K]; labels y [T] (int64, shifted).

    The input gradient is computed in forward, chunk by chunk: logits = h_c W^T (bf16), the loss kernel overwrites
    them with d loss / d logits, dh_c = dlogits W.  Only one chunk of bf16 logits exists at a time and no fp32 logits at
    all; the saved state is dh [T, K].  Backward returns dh * grad_output (exact for grad_output == 1).

    The fused forward GEMM takes whole N tiles of 256; for V % 256 != 0 (Qwen3: 151 936 = 593 * 256 + 128) it writes
    the first V - V % 256 columns of each chunk and one library GEMM fills the last V % 256 (under 0.1 % of the work
    at Qwen3's vocabulary)."""

    @staticmethod
    def forward(ctx, h, weight, labels, denom, ignore_index):
        T = h.shape[0]
        V = weight.shape[0]
        V0 = V - V % _LM_HEAD_TILE_N
        scale = denom.float().reciprocal().reshape(1)      # the fp32 1/denom autograd of HF's loss propagates
        loss_rows = torch.empty(T, dtype=torch.float32, device=h.device)
        dh = torch.empty_like(h)
        for s in range(0, T, _CE_CHUNK_ROWS):
            e = min(T, s + _CE_CHUNK_ROWS)
            if V0 == V:
                logits = ops.fused_linear_forward(h[s:e], [weight])[0]
            else:
                logits = torch.empty(e - s, V, dtype=h.dtype, device=h.device)
                ops.fused_linear_forward(h[s:e], [weight[:V0]], out=logits[:, :V0])
                torch.mm(h[s:e], weight[V0:].t(), out=logits[:, V0:])
            loss_rows[s:e] = ops.cross_entropy_rows(logits, labels[s:e], scale, ignore_index)
            ops.fused_linear_dgrad([logits], [weight], out=dh[s:e])
            del logits
        ctx.save_for_backward(dh)
        return loss_rows.sum() / denom

    @staticmethod
    def backward(ctx, grad_output):
        dh, = ctx.saved_tensors
        return dh * grad_output, None, None, None, None


def causal_lm_loss(h, weight, labels, ignore_index=-100, shift_labels=None, num_items_in_batch=None, **_):
    """transformers' `ForCausalLMLoss(h @ weight.T, labels, ...)` through `LinearCrossEntropyFn`: labels shifted (or
    `shift_labels` as given), mean over the labels that are not `ignore_index`, or sum / `num_items_in_batch`."""
    if shift_labels is None:
        labels = nn.functional.pad(labels, (0, 1), value=ignore_index)
        shift_labels = labels[..., 1:]
    y = shift_labels.reshape(-1).to(device=h.device, dtype=torch.int64).contiguous()
    h2 = h.reshape(-1, h.shape[-1]).contiguous()
    if num_items_in_batch is None:
        denom = (y != ignore_index).sum()                   # on the device: no host sync
    else:
        denom = torch.as_tensor(num_items_in_batch, device=h.device)
    return LinearCrossEntropyFn.apply(h2, weight, y, denom, int(ignore_index))


# ---- when the native path applies ------------------------------------------------------------------------------------

_MAX_NORM_WIDTH = 32768     # smt_rmsnorm_*: up to 4 x 1024 16-byte vectors per row
_hf_only = threading.local()


class _plain_hf:
    """Inside: every override runs its class's own forward (a layer that fell back takes its submodules with it)."""

    def __enter__(self):
        _hf_only.depth = getattr(_hf_only, "depth", 0) + 1

    def __exit__(self, *exc):
        _hf_only.depth -= 1
        return False


def _native(*ts) -> bool:
    if getattr(_hf_only, "depth", 0):
        return False
    return all(t.is_cuda and t.dtype == torch.bfloat16 for t in ts)


def _norm_ok(norm, x) -> bool:
    w = norm.weight
    return _native(x, w) and not w.requires_grad and w.dim() == 1 and x.shape[-1] == w.shape[0] \
        and w.shape[0] % 8 == 0 and w.shape[0] <= _MAX_NORM_WIDTH and w.is_contiguous() and w.data_ptr() % 16 == 0


def _rope_ok(q, k, cos, sin) -> bool:
    # q, k: [B, S, H, 128] views of the projections' outputs; cos / sin: [1 or B, S, 128] rows of 128
    return _native(q, k, cos, sin) and q.dim() == 4 and q.shape[-1] == 128 and k.shape[-1] == 128 \
        and q.is_contiguous() and k.is_contiguous() and cos.dim() == 3 and cos.shape == sin.shape \
        and cos.shape[1:] == (q.shape[1], 128) and cos.shape[0] in (1, q.shape[0]) \
        and cos.stride() == sin.stride() and cos.stride()[1:] == (128, 1)


# ---- the overrides (bodies follow transformers' modeling_llama) ---------------------------------------------------

def _rmsnorm_forward(self, hidden_states):
    if _norm_ok(self, hidden_states):
        return RMSNormFn.apply(hidden_states.contiguous(), self.weight, float(self.variance_epsilon))
    return type(self).forward(self, hidden_states)


def _mlp_forward(self, x):
    if getattr(_hf_only, "depth", 0):
        return type(self).forward(self, x)
    g, u = self.gate_proj(x), self.up_proj(x)
    if _native(g, u) and g.shape == u.shape and g.numel() % 8 == 0:
        h = SwiGLUFn.apply(g.contiguous(), u.contiguous())
    else:
        h = self.act_fn(g) * u
    return self.down_proj(h)


def _qk_norms_ok(attn) -> bool:
    # Qwen3's per-head norms: frozen bf16 weights of width 128 that the kernel can read directly
    return all(not n.weight.requires_grad and _native(n.weight) and n.weight.shape == (128,)
               and n.weight.is_contiguous() and n.weight.data_ptr() % 16 == 0 for n in (attn.q_norm, attn.k_norm))


def _attention_forward(self, hidden_states, position_embeddings=None, attention_mask=None, past_key_values=None,
                       **kwargs):
    F = _family_of(self, "Attention")
    if past_key_values is not None or position_embeddings is None or getattr(_hf_only, "depth", 0) \
            or (F.qk_norm and (self.q_norm.weight.requires_grad or self.k_norm.weight.requires_grad)):
        return type(self).forward(self, hidden_states, position_embeddings, attention_mask, past_key_values, **kwargs)
    L = F.modeling()
    input_shape = hidden_states.shape[:-1]
    hidden_shape = (*input_shape, -1, self.head_dim)

    query_states = self.q_proj(hidden_states).view(hidden_shape)
    key_states = self.k_proj(hidden_states).view(hidden_shape)
    value_states = self.v_proj(hidden_states).view(hidden_shape).transpose(1, 2)

    cos, sin = position_embeddings
    if _rope_ok(query_states, key_states, cos, sin) and (not F.qk_norm or _qk_norms_ok(self)):
        # outputs in the projections' [B, S, H, D] layout, handed on as [B, H, S, D] views: the strides HF's
        # elementwise RoPE produces, so the attention kernel is fed exactly as before
        if F.qk_norm:
            query_states, key_states = QKNormRoPEFn.apply(
                query_states, key_states, self.q_norm.weight, self.k_norm.weight, float(self.q_norm.variance_epsilon),
                float(self.k_norm.variance_epsilon), cos, sin)
        else:
            query_states, key_states = RoPEFn.apply(query_states, key_states, cos, sin)
        query_states, key_states = query_states.transpose(1, 2), key_states.transpose(1, 2)
    else:
        if F.qk_norm:
            query_states, key_states = self.q_norm(query_states), self.k_norm(key_states)
        query_states, key_states = L.apply_rotary_pos_emb(query_states.transpose(1, 2), key_states.transpose(1, 2),
                                                          cos, sin)

    attention_interface = L.ALL_ATTENTION_FUNCTIONS.get_interface(self.config._attn_implementation,
                                                                  L.eager_attention_forward)
    attn_output, attn_weights = attention_interface(
        self,
        query_states,
        key_states,
        value_states,
        attention_mask,
        dropout=0.0 if not self.training else self.attention_dropout,
        scaling=self.scaling,
        **F.attention_kwargs(self),
        **kwargs,
    )
    attn_output = attn_output.reshape(*input_shape, -1).contiguous()
    attn_output = self.o_proj(attn_output)
    return attn_output, attn_weights


def _decoder_forward(self, hidden_states, attention_mask=None, position_ids=None, past_key_values=None, use_cache=False,
                     position_embeddings=None, **kwargs):
    args = dict(attention_mask=attention_mask, position_ids=position_ids, past_key_values=past_key_values,
                use_cache=use_cache, position_embeddings=position_embeddings, **kwargs)
    if past_key_values is not None:
        with _plain_hf():
            return type(self).forward(self, hidden_states, **args)
    post_norm = self.post_attention_layernorm
    if not _norm_ok(post_norm, hidden_states):
        return type(self).forward(self, hidden_states, **args)
    residual = hidden_states
    hidden_states = self.input_layernorm(hidden_states)
    hidden_states, _ = self.self_attn(hidden_states=hidden_states, **args)
    if _native(hidden_states) and hidden_states.shape == residual.shape:
        residual, hidden_states = AddRMSNormFn.apply(residual.contiguous(), hidden_states.contiguous(), post_norm.weight,
                                                     float(post_norm.variance_epsilon))
    else:
        residual = residual + hidden_states
        hidden_states = post_norm(residual)
    hidden_states = self.mlp(hidden_states)
    return residual + hidden_states


def _lm_head_ok(model, h) -> bool:
    head = model.lm_head
    if type(head) is not nn.Linear or head.bias is not None:
        return False
    w = head.weight
    V0 = w.shape[0] - w.shape[0] % _LM_HEAD_TILE_N           # columns the fused forward GEMM computes
    return _native(h, w) and h.requires_grad and not w.requires_grad and w.shape[0] == model.config.vocab_size \
        and h.shape[-1] == w.shape[1] and w.shape[0] % 8 == 0 and V0 > 0 and ops.fused_linear_supported([w[:V0]]) \
        and ops.fused_linear_supported([w], dgrad=True)


def _causal_lm_forward(self, input_ids=None, attention_mask=None, position_ids=None, past_key_values=None,
                       inputs_embeds=None, labels=None, use_cache=None, logits_to_keep=0, **kwargs):
    args = dict(input_ids=input_ids, attention_mask=attention_mask, position_ids=position_ids,
                past_key_values=past_key_values, inputs_embeds=inputs_embeds, use_cache=use_cache)
    if labels is None or not isinstance(logits_to_keep, int) or logits_to_keep != 0 or past_key_values is not None \
            or not torch.is_grad_enabled() or getattr(_hf_only, "depth", 0):
        return type(self).forward(self, **args, labels=labels, logits_to_keep=logits_to_keep, **kwargs)
    # `return_dict` as transformers' `can_return_tuple` resolves it
    return_dict = self.config.return_dict if hasattr(self, "config") else True
    passed = kwargs.pop("return_dict", return_dict)
    if passed is not None:
        return_dict = passed
    outputs = self.model(**args, **kwargs)
    h = outputs.last_hidden_state
    if outputs.past_key_values is None and self.loss_function is _causal_lm_loss_fn() and _lm_head_ok(self, h):
        loss = causal_lm_loss(h, self.lm_head.weight, labels, **kwargs)
        logits = None
    else:
        logits = self.lm_head(h)
        loss = self.loss_function(logits=logits, labels=labels, vocab_size=self.config.vocab_size, **kwargs)
    from transformers.modeling_outputs import CausalLMOutputWithPast
    out = CausalLMOutputWithPast(loss=loss, logits=logits, past_key_values=outputs.past_key_values,
                                 hidden_states=outputs.hidden_states, attentions=outputs.attentions)
    return out if return_dict else out.to_tuple()


# ---- model families, version guard and installation ------------------------------------------------------------------

# Forward signatures the overrides copy, by role; LLaMA, Mistral and Qwen3 share them in the transformers version this
# module was written against.
_EXPECTED_PARAMS = {
    "RMSNorm": ["self", "hidden_states"],
    "MLP": ["self", "x"],
    "Attention": ["self", "hidden_states", "position_embeddings", "attention_mask", "past_key_values", "kwargs"],
    "DecoderLayer": ["self", "hidden_states", "attention_mask", "position_ids", "past_key_values", "use_cache",
                     "position_embeddings", "kwargs"],
    "ForCausalLM": ["self", "input_ids", "attention_mask", "position_ids", "past_key_values", "inputs_embeds",
                    "labels", "use_cache", "logits_to_keep", "kwargs"],
}


class _Family:
    """One transformers model family whose decoder the overrides reproduce: its modeling module, class-name prefix
    (`<prefix>DecoderLayer`, ...), the keyword arguments its attention body adds to the attention interface call, and
    whether q / k pass through a per-head RMSNorm (`q_norm` / `k_norm`) before RoPE."""

    def __init__(self, name, prefix, attention_kwargs, qk_norm):
        self.name, self.prefix, self.attention_kwargs, self.qk_norm = name, prefix, attention_kwargs, qk_norm
        self._mod = None

    def modeling(self):
        if self._mod is None:
            import importlib
            self._mod = importlib.import_module(f"transformers.models.{self.name}.modeling_{self.name}")
        return self._mod


_FAMILIES = (
    _Family("llama", "Llama", lambda attn: {}, qk_norm=False),
    _Family("mistral", "Mistral", lambda attn: {"sliding_window": getattr(attn.config, "sliding_window", None)},
            qk_norm=False),
    _Family("qwen3", "Qwen3", lambda attn: {"sliding_window": attn.sliding_window}, qk_norm=True),
)
_family_cache = {}


def _causal_lm_loss_fn():
    from transformers.loss.loss_utils import ForCausalLMLoss
    return ForCausalLMLoss


def _class_matches(module, family: _Family, role: str) -> bool:
    """`module` is exactly `family`'s transformers class for `role`, whose forward has the signature these overrides
    copy."""
    try:
        cls = getattr(family.modeling(), family.prefix + role)
    except (ImportError, AttributeError):
        return False
    return type(module) is cls and list(inspect.signature(cls.forward).parameters) == _EXPECTED_PARAMS[role]


def _family_of(module, role: str):
    """The family whose class for `role` `module` is exactly, or None."""
    key = (type(module), role)
    if key not in _family_cache:
        _family_cache[key] = next((f for f in _FAMILIES if _class_matches(module, f, role)), None)
    return _family_cache[key]


def layer_supported(layer) -> bool:
    """A LLaMA, Mistral or Qwen3 decoder layer of the transformers version this module was written against, with
    head_dim 128 and a SiLU MLP (Qwen3: q_norm / k_norm of width 128)."""
    F = _family_of(layer, "DecoderLayer")
    if F is None:
        return False
    attn, mlp = getattr(layer, "self_attn", None), getattr(layer, "mlp", None)
    norms = (getattr(layer, "input_layernorm", None), getattr(layer, "post_attention_layernorm", None))
    if not (_class_matches(attn, F, "Attention") and _class_matches(mlp, F, "MLP")
            and all(_class_matches(n, F, "RMSNorm") for n in norms) and getattr(attn, "head_dim", None) == 128
            and type(mlp.act_fn).__name__ in ("SiLUActivation", "SiLU")):
        return False
    if F.qk_norm:
        qk = (getattr(attn, "q_norm", None), getattr(attn, "k_norm", None))
        return all(_class_matches(n, F, "RMSNorm") and tuple(n.weight.shape) == (128,) for n in qk)
    return True


def install_layer(layer) -> bool:
    """Install the overrides on one decoder layer (see the module docstring); False when the layer is unsupported."""
    if not layer_supported(layer):
        return False
    install_forward(layer, _decoder_forward)
    install_forward(layer.self_attn, _attention_forward)
    install_forward(layer.mlp, _mlp_forward)
    install_forward(layer.input_layernorm, _rmsnorm_forward)
    install_forward(layer.post_attention_layernorm, _rmsnorm_forward)
    return True


def install_norm(norm) -> bool:
    """The RMSNorm override alone (a model's final norm)."""
    if _family_of(norm, "RMSNorm") is None:
        return False
    install_forward(norm, _rmsnorm_forward)
    return True


def install_causal_lm(model) -> bool:
    """The fused lm_head + causal-LM loss override on a `LlamaForCausalLM`, `MistralForCausalLM` or `Qwen3ForCausalLM`;
    False for any other class."""
    if _family_of(model, "ForCausalLM") is None:
        return False
    install_forward(model, _causal_lm_forward)
    return True


def remove_causal_lm(model) -> bool:
    """Undo `install_causal_lm`; False when the model had no such override."""
    if getattr(model.__dict__.get("forward"), "__func__", None) is not _causal_lm_forward:
        return False
    return remove_forward(model)


def remove_all(model) -> int:
    """Remove every override `install_layer` / `install_norm` installed under `model`; returns the number of layers."""
    n = 0
    for mod in model.modules():
        fn = getattr(mod.__dict__.get("forward"), "__func__", None)
        if fn in _OVERRIDES:
            remove_forward(mod)
            n += fn is _decoder_forward
    return n


_OVERRIDES = (_decoder_forward, _attention_forward, _mlp_forward, _rmsnorm_forward)
