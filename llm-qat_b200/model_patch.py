"""Opt-in acceleration of the callers either side of the fake-quant path (SURVEY.md section 8f), for a
model built from the reference's UNMODIFIED ``models/modeling_llama_quant.py`` (or the harness that
mirrors it):

    import llm_qat_b200; llm_qat_b200.install()
    from models.modeling_llama_quant import LlamaForCausalLM
    model = LlamaForCausalLM(config).bfloat16().cuda()
    llm_qat_b200.fuse_model(model)          # default off: without this call nothing below is active

``fuse_model`` rebinds ``forward`` on module INSTANCES (found by their attributes, not by class), so the
model file, its classes, parameters and state dict are untouched and ``unfuse_model`` restores them:

* attention (q_proj/k_proj/v_proj/o_proj + rotary_emb; modeling_llama_quant.py:301-393): three
  QuantizeLinear GEMMs sharing one set of activation codes -> ONE kernel for the K/V per-token fake-quant
  (:320-327) and RoPE (:334-341) -> the tcgen05 causal attention kernel (:352-377) -> o_proj.  Taken only
  when the additive mask is the causal mask the model itself built (:60-92,:599-629), head_dim == 128 and
  the tensors are bf16; anything else (padding masks, past_key_value, output_attentions, other dtypes)
  runs the reference's own forward.
* MLP (:234-235): silu(gate) * up in one kernel that also emits down_proj's activation codes.
* RMSNorm (:121-129): one kernel that also emits the codes q/k/v (or gate/up) consume.
* QuantizeLinear off the int8 grid (W4-A16, weight-only QAT with W1/W2, 9..31-bit weights, activation-only):
  the reference's exact bf16 operands, from one K1 pass each, contracted on this library's tcgen05 GEMM
  forward and backward (utils_quant._OperandLinearFn).  Marked per instance (``_qat_operand_route``); the
  int8-grid configurations keep their own path either way.
* ``fuse_kd_loss(trainer)``: KDTrainer.ce_loss (utils/kd_trainer.py:42-48) -> fused_ops.kd_loss.
"""
from __future__ import annotations

import collections
import types

import torch

from . import fused_ops as F
from .utils_quant import QuantizeLinear, SymQuantizer, _clip_bounds, operand_route_config

__all__ = ["fuse_model", "unfuse_model", "fuse_kd_loss", "mark_causal_mask"]

# The additive causal masks most recently built by fused models (strong references: a registered mask's
# storage cannot be recycled for another tensor).  Attention treats a mask as causal iff it IS one of these
# storages.  More than one is kept because a step holds more than one model's mask at a time — the FP
# teacher's and the student's (kd_trainer.py:53-64), whose checkpoint recompute presents the student's mask
# again during backward — and the recompute must take the same path as the forward it repeats, whatever
# the order of the two forwards.  [b, 1, s, s] bf16 at s = 2048 is 8 MB per entry.
_CAUSAL_KEEP = 4
_CAUSAL: collections.deque = collections.deque(maxlen=_CAUSAL_KEEP)


def mark_causal_mask(mask: torch.Tensor) -> torch.Tensor:
    """Declare ``mask`` ([b, 1, s, s] additive, finfo.min above the diagonal, 0 elsewhere — what
    ``_make_causal_mask`` builds, modeling_llama_quant.py:60-92) as purely causal."""
    if not _is_causal(mask):
        _CAUSAL.append(mask)
    return mask


def _is_causal(mask) -> bool:
    if mask is None:
        return False
    ptr = mask.data_ptr()
    for ref in tuple(_CAUSAL):      # a snapshot: autograd's backward thread may look while a forward registers
        if (ptr == ref.data_ptr() and mask.shape == ref.shape and mask.dtype == ref.dtype
                and mask.device == ref.device):
            return True
    return False


def _fusable_linear(lin) -> int:
    """a_bits when ``lin`` is a QuantizeLinear whose forward takes the integer-grid path, else 0."""
    if isinstance(lin, QuantizeLinear) and 3 <= lin.w_bits <= 8 and 3 <= lin.a_bits <= 8 \
            and getattr(lin, "act_quantizer", None) is SymQuantizer and not lin.act_layerwise \
            and not lin.weight_layerwise and lin.in_features % 16 == 0:
        return int(lin.a_bits)
    return 0


# ---------------------------------------------------------------------------------- attention
def _rope_tables(self, seq_len: int, device):
    """fp32 [max_pos, head_dim] cos / sin tables of the module's rotary embedding (:132-171)."""
    rot = self.rotary_emb
    if seq_len > rot.cos_cached.shape[2]:
        return None, None
    tabs = getattr(self, "_qat_rope", None)
    if tabs is None or tabs[0].device != device:
        cos = rot.cos_cached[0, 0].to(device=device, dtype=torch.float32).contiguous()
        sin = rot.sin_cached[0, 0].to(device=device, dtype=torch.float32).contiguous()
        tabs = (cos, sin)
        self._qat_rope = tabs
    return tabs


def _on_gpu(t: torch.Tensor) -> bool:
    """The fused kernels exist for CUDA tensors only (tests substitute CPU emulations and patch this)."""
    return t.is_cuda


def _module_clip(self):
    """(lo, hi) of act_clip_val_k, read once per tensor version: a clip tensor that lives on the GPU (a model
    built under `with torch.device("cuda")`) would otherwise cost a device-to-host sync in every forward."""
    t = getattr(self, "act_clip_val_k", None)
    if t is None:
        return (-2.0, 2.0)
    key = (id(t), t._version)
    cached = self.__dict__.get("_qat_clip")
    if cached is None or cached[0] != key:
        cached = (key, _clip_bounds(t))
        self.__dict__["_qat_clip"] = cached
    return cached[1]


def _attention_forward(self, hidden_states, attention_mask=None, position_ids=None, past_key_value=None,
                       output_attentions=False, use_cache=False):
    orig = self._qat_orig_forward
    if (past_key_value is not None or output_attentions or position_ids is None or self.head_dim != 128
            or not _on_gpu(hidden_states) or not _is_causal(attention_mask)):
        return orig(hidden_states, attention_mask, position_ids, past_key_value, output_attentions, use_cache)
    # the projections return the autocast dtype inside torch.autocast, else their input's: decide BEFORE running
    # them, so that a model in another dtype (fp32, fp16) does not compute q/k/v twice
    proj_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else hidden_states.dtype
    if proj_dtype != torch.bfloat16:
        return orig(hidden_states, attention_mask, position_ids, past_key_value, output_attentions, use_cache)
    bsz, q_len, _ = hidden_states.size()
    cos, sin = _rope_tables(self, q_len, hidden_states.device)
    if cos is None:
        return orig(hidden_states, attention_mask, position_ids, past_key_value, output_attentions, use_cache)
    q = self.q_proj(hidden_states)
    k = self.k_proj(hidden_states)
    v = self.v_proj(hidden_states)
    if q.dtype != torch.bfloat16 or k.dtype != torch.bfloat16 or v.dtype != torch.bfloat16:
        # not reached with the reference's modules (see above); a foreign projection class that returns another
        # dtype: take the reference path (it recomputes the projections)
        return orig(hidden_states, attention_mask, position_ids, past_key_value, output_attentions, use_cache)
    pos = position_ids.expand(bsz, q_len) if position_ids.shape[0] != bsz else position_ids
    kv_bits = int(getattr(self, "kv_bits", 32))     # a stock (teacher) LlamaAttention has no K/V fake-quant
    clip = _module_clip(self)
    qr, kr, vq = F.qkv_prep(q, k, v, cos, sin, pos, self.num_heads, kv_bits, clip)
    shape = (bsz, q_len, self.num_heads, self.head_dim)
    o = F.causal_attention(qr.view(shape), kr.view(shape), vq.view(shape), causal=True)
    out = self.o_proj(o.reshape(bsz, q_len, self.hidden_size))
    present = (kr.view(shape).transpose(1, 2), vq.view(shape).transpose(1, 2)) if use_cache else None
    return out, None, present


# ---------------------------------------------------------------------------------- MLP, RMSNorm
def _is_silu(fn) -> bool:
    return fn is torch.nn.functional.silu or isinstance(fn, torch.nn.SiLU) or type(fn).__name__ in ("SiLUActivation", "SiLU")


def _mlp_forward(self, x):
    gate = self.gate_proj(x)
    up = self.up_proj(x)
    if not F.swiglu_supported(gate, up):
        return self.down_proj(self.act_fn(gate) * up)
    return self.down_proj(F.swiglu(gate, up, feed_bits=self._qat_feed_bits))


def _rmsnorm_forward(self, hidden_states):
    if not F.rmsnorm_supported(hidden_states, self.weight):
        return self._qat_orig_forward(hidden_states)
    return F.rmsnorm(hidden_states, self.weight, self.variance_epsilon, feed_bits=self._qat_feed_bits)


# ---------------------------------------------------------------------------------- the model's mask
def _model_forward(self, *args, **kwargs):
    am = kwargs.get("attention_mask", args[1] if len(args) > 1 else None)
    # None is what the recipe's dataset gives (utils/datautils.py returns input_ids / labels only) and the
    # model then builds an all-ones mask itself (:672-675); an explicit mask costs one small sync here
    self._qat_plain_causal = am is None or bool(am.to(torch.bool).all())
    return self._qat_orig_forward(*args, **kwargs)


def _prepare_mask(self, attention_mask, input_shape, inputs_embeds, past_key_values_length):
    m = self._qat_orig_prepare(attention_mask, input_shape, inputs_embeds, past_key_values_length)
    if getattr(self, "_qat_plain_causal", False) and past_key_values_length == 0 and m is not None:
        mark_causal_mask(m)
    return m     # a padded / cached-prefix mask is simply never registered: its calls run the reference's attention


def _bind(mod, name, fn):
    if not hasattr(mod, "_qat_orig_" + name):
        setattr(mod, "_qat_orig_" + name, getattr(mod, name))
    setattr(mod, name, types.MethodType(fn, mod))


def fuse_model(model, attention: bool = True, mlp: bool = True, rmsnorm: bool = True, linear: bool = True):
    """Rebind the forward of every attention / MLP / RMSNorm module of ``model`` and, with ``linear``, mark the
    QuantizeLinear modules the operand route serves (see module docstring; ``linear=False`` clears the marks).
    Returns the model.  Idempotent."""
    for mod in model.modules():
        if isinstance(mod, QuantizeLinear):
            if linear and operand_route_config(mod):
                mod._qat_operand_route = True
            else:
                mod.__dict__.pop("_qat_operand_route", None)
        has = lambda *names: all(hasattr(mod, n) for n in names)  # noqa: E731
        if attention and has("q_proj", "k_proj", "v_proj", "o_proj", "rotary_emb", "num_heads", "head_dim"):
            _bind(mod, "forward", _attention_forward)
        elif mlp and has("gate_proj", "up_proj", "down_proj", "act_fn") and _is_silu(mod.act_fn):
            mod._qat_feed_bits = _fusable_linear(mod.down_proj)
            _bind(mod, "forward", _mlp_forward)
        elif has("_prepare_decoder_attention_mask", "layers", "embed_tokens"):
            _bind(mod, "forward", _model_forward)
            if not hasattr(mod, "_qat_orig_prepare"):
                mod._qat_orig_prepare = mod._prepare_decoder_attention_mask
            mod._prepare_decoder_attention_mask = types.MethodType(_prepare_mask, mod)
        if rmsnorm and has("self_attn", "mlp", "input_layernorm", "post_attention_layernorm"):
            for norm, consumer in ((mod.input_layernorm, getattr(mod.self_attn, "q_proj", None)),
                                   (mod.post_attention_layernorm, getattr(mod.mlp, "gate_proj", None))):
                if hasattr(norm, "variance_epsilon") and hasattr(norm, "weight"):
                    norm._qat_feed_bits = _fusable_linear(consumer)
                    _bind(norm, "forward", _rmsnorm_forward)
    if rmsnorm:   # norms outside a decoder layer (the model's final norm feeds the plain lm_head): no codes
        for mod in model.modules():
            if hasattr(mod, "variance_epsilon") and hasattr(mod, "weight") and "_qat_orig_forward" not in mod.__dict__:
                mod._qat_feed_bits = 0
                _bind(mod, "forward", _rmsnorm_forward)
    return model


def unfuse_model(model):
    for mod in model.modules():
        mod.__dict__.pop("_qat_operand_route", None)
        if "_qat_orig_forward" in mod.__dict__:
            del mod.forward                    # the instance attribute; the class's forward shows again
            del mod._qat_orig_forward
        if "_qat_orig_prepare" in mod.__dict__:
            del mod._prepare_decoder_attention_mask
            del mod._qat_orig_prepare
    return model


def fuse_kd_loss(trainer):
    """KDTrainer.ce_loss (utils/kd_trainer.py:42-48) -> the fused KL kernel (one pass per direction)."""
    trainer.ce_loss = lambda student_logits, teacher_logits: F.kd_loss(student_logits, teacher_logits)
    return trainer
