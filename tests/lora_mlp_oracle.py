"""fp32 CPU reference of LoRA adapters on any subset of q/k/v/gate/up/down_proj.  TEST INFRASTRUCTURE ONLY.

oracle/llama_lora.py restates the training step with adapters on the attention projections; this module extends its forward
pass to the MLP projections and reuses everything else (RMSNorm, RoPE, attention, dropout masks, loss, AdamW):
  * peft 0.5.0 lora.Linear on every enabled module: y = x W^T + (alpha/r) * B A dropout(x), one independent dropout per module;
  * mlp.gate_proj / mlp.up_proj take h2 = post_attention_layernorm(x) [M, hidden]: lora_A [r, hidden], lora_B [ffn, r];
  * mlp.down_proj takes act = silu(gate) * up [M, ffn]: lora_A [r, ffn], lora_B [hidden, r];
  * lora_A ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)), lora_B = 0;
  * the dropout mask of a module is indexed by its position among the enabled targets in HF module order
    (q, k, v, gate, up, down) and has the module's input width (ffn for down_proj).
For q/k/v-only configurations every function here computes exactly what oracle/llama_lora.py computes.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from oracle import llama_lora as O

LORA_MODULES = ("q_proj", "k_proj", "v_proj", "gate_proj", "up_proj", "down_proj")
MLP_MODULES = ("gate_proj", "up_proj", "down_proj")


def module_path(target: str) -> str:
    """Path of a linear module inside a decoder layer (modeling_llama.py LlamaAttention / LlamaMLP)."""
    return f"mlp.{target}" if target in MLP_MODULES else f"self_attn.{target}"


def linear_dims(cfg: O.OracleConfig, target: str) -> Tuple[int, int]:
    """(in, out) features of a decoder layer's linear module."""
    d, F = cfg.hidden, cfg.ffn
    dkv = (cfg.n_kv_heads or cfg.n_heads) * cfg.head_dim
    return {"q_proj": (d, d), "k_proj": (d, dkv), "v_proj": (d, dkv), "gate_proj": (d, F), "up_proj": (d, F), "down_proj": (F, d)}[target]


def init_lora(cfg: O.OracleConfig, seed: int = 4321) -> Dict[str, torch.Tensor]:
    """peft 0.5.0 LoraLayer.reset_lora_parameters with each module's own fan-in (the same generator stream as O.init_lora)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    r = cfg.lora_r
    for l in range(cfg.n_layers):
        for t in cfg.lora_target:
            d_in, d_out = linear_dims(cfg, t)
            bound = 1.0 / math.sqrt(d_in)
            p = f"model.layers.{l}.{module_path(t)}."
            out[p + "lora_A.weight"] = (torch.rand(r, d_in, generator=g) * 2 - 1) * bound
            out[p + "lora_B.weight"] = torch.zeros(d_out, r)
    return out


def dropout_masks(cfg: O.OracleConfig, drop_ctx: Optional[Tuple[int, int]], layer: int, n_rows: int) -> Dict[str, torch.Tensor]:
    """The keep masks of one layer's enabled targets, {} without dropout."""
    if drop_ctx is None or cfg.lora_dropout <= 0:
        return {}
    key = O.dropout_key(cfg.seed, drop_ctx[0], layer, drop_ctx[1])
    targets = [t for t in LORA_MODULES if t in cfg.lora_target]
    return {t: O.dropout_mask(key, i, n_rows, linear_dims(cfg, t)[0], cfg.lora_dropout) for i, t in enumerate(targets)}


def forward_logits(cfg: O.OracleConfig, w: Dict[str, torch.Tensor], lora: Dict[str, torch.Tensor], ids: torch.Tensor,
                   drop_ctx: Optional[Tuple[int, int]] = None) -> torch.Tensor:
    """O.forward_logits with adapters on every enabled module (drop_ctx = (fwd_count, rank) enables dropout)."""
    B, S = ids.shape
    H, D = cfg.n_heads, cfg.head_dim
    Hkv = cfg.n_kv_heads or H
    scale = cfg.lora_alpha / cfg.lora_r
    cos, sin = O.rope_cos_sin(S, D, cfg.rope_theta)
    x = w["model.embed_tokens.weight"][ids.long()]
    for l in range(cfg.n_layers):
        p = f"model.layers.{l}."
        masks = dropout_masks(cfg, drop_ctx, l, B * S)

        def proj(name, inp):
            m = p + module_path(name)
            a, b = lora.get(m + ".lora_A.weight"), lora.get(m + ".lora_B.weight")
            return O.lora_linear(inp, w[m + ".weight"], a, b, scale, masks.get(name) if a is not None else None, cfg.lora_dropout)

        h = O.rmsnorm(x, w[p + "input_layernorm.weight"], cfg.rms_eps)
        q = proj("q_proj", h).view(B, S, H, D).transpose(1, 2)
        k = proj("k_proj", h).view(B, S, Hkv, D).transpose(1, 2)
        v = proj("v_proj", h).view(B, S, Hkv, D).transpose(1, 2)
        q, k = O.apply_rope(q, cos, sin), O.apply_rope(k, cos, sin)
        if Hkv != H:
            k = k.repeat_interleave(H // Hkv, dim=1)
            v = v.repeat_interleave(H // Hkv, dim=1)
        o = O.attention(q, k, v, cfg.sliding_window if S > cfg.sliding_window + 1 else 0).transpose(1, 2).reshape(B, S, H * D)
        x = x + o @ w[p + "self_attn.o_proj.weight"].t()
        h2 = O.rmsnorm(x, w[p + "post_attention_layernorm.weight"], cfg.rms_eps)
        act = torch.nn.functional.silu(proj("gate_proj", h2)) * proj("up_proj", h2)
        x = x + proj("down_proj", act)
    x = O.rmsnorm(x, w["model.norm.weight"], cfg.rms_eps)
    return (x @ w["lm_head.weight"].t()).float()


class OracleTrainer(O.OracleTrainer):
    """O.OracleTrainer (gradient mean, clipping, AdamW, schedule, dropout-key bookkeeping) over forward_logits above."""

    def loss_and_grads(self, ids: np.ndarray, labels: np.ndarray, rank: int = 0,
                       fwd_count: Optional[int] = None) -> Tuple[float, Dict[str, torch.Tensor]]:
        for p in self.lora.values():
            p.grad = None
        if fwd_count is None:
            self.fwd_count += 1
            fwd_count = self.fwd_count
        logits = forward_logits(self.cfg, self.w, self.lora, torch.from_numpy(np.asarray(ids)).long(), (fwd_count, rank))
        loss = O.causal_lm_loss(logits, torch.from_numpy(np.asarray(labels)).long())
        loss.backward()
        return float(loss.detach()), {k: p.grad.detach().clone() for k, p in self.lora.items()}

    def eval_loss(self, ids: np.ndarray, labels: np.ndarray) -> float:
        self.fwd_count += 1
        with torch.no_grad():
            logits = forward_logits(self.cfg, self.w, self.lora, torch.from_numpy(np.asarray(ids)).long())
            return float(O.causal_lm_loss(logits, torch.from_numpy(np.asarray(labels)).long()))
