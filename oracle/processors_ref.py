"""CPU oracle: restatement of the reference's two attention processors.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  PINNED against the reference
itself: tests/golden/ holds outputs of the reference attention.py imported
verbatim (via oracle/diffusers_shim) by tests/golden/make_golden.py and
tests/golden/make_pinned_golden.py, and tests/test_oracle_cpu.py compares.

Follows:
  attention.py:90-174   Consistent_AttProcessor   (LoRA'd self-attention; without xformers
                        the core is ``attn.get_attention_scores`` + ``bmm``, :156-158)
  attention.py:177-294  Consistent_IPAttProcessor (LoRA'd text cross-attention + decoupled
                        4-token ID branch: two softmaxes sharing Q, ``o_text + scale*o_ip``, :259-279)
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F


class LoRALinearRef(nn.Module):
    """diffusers 0.23 ``LoRALinearLayer`` (used at attention.py:105-108, 194-197)."""

    def __init__(self, in_features, out_features, rank, network_alpha=None):
        super().__init__()
        self.down = nn.Linear(in_features, rank, bias=False)
        self.up = nn.Linear(rank, out_features, bias=False)
        self.network_alpha, self.rank = network_alpha, rank
        nn.init.normal_(self.down.weight, std=1.0 / rank)
        nn.init.zeros_(self.up.weight)

    def forward(self, x):
        y = self.up(self.down(x.to(self.down.weight.dtype)))
        if self.network_alpha is not None:
            y = y * (self.network_alpha / self.rank)
        return y.to(x.dtype)


def _flatten_spatial(x):
    if x.ndim == 4:
        b, c, h, w = x.shape
        return x.view(b, c, h * w).transpose(1, 2), (b, c, h, w)
    return x, None


def _finish(attn, y, residual, shape4):
    if shape4 is not None:
        b, c, h, w = shape4
        y = y.transpose(-1, -2).reshape(b, c, h, w)
    if attn.residual_connection:
        y = y + residual
    return y / attn.rescale_output_factor


class ConsistentAttnRef(nn.Module):
    def __init__(self, hidden_size=None, cross_attention_dim=None, rank=4, network_alpha=None, lora_scale=1.0):
        super().__init__()
        self.rank, self.lora_scale = rank, lora_scale
        kv_in = cross_attention_dim or hidden_size
        self.to_q_lora = LoRALinearRef(hidden_size, hidden_size, rank, network_alpha)
        self.to_k_lora = LoRALinearRef(kv_in, hidden_size, rank, network_alpha)
        self.to_v_lora = LoRALinearRef(kv_in, hidden_size, rank, network_alpha)
        self.to_out_lora = LoRALinearRef(hidden_size, hidden_size, rank, network_alpha)

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None):
        residual = hidden_states
        x, shape4 = _flatten_spatial(hidden_states)
        s = self.lora_scale
        ctx = x if encoder_hidden_states is None else encoder_hidden_states
        q = attn.to_q(x) + s * self.to_q_lora(x)
        k = attn.to_k(ctx) + s * self.to_k_lora(ctx)
        v = attn.to_v(ctx) + s * self.to_v_lora(ctx)
        q, k, v = (attn.head_to_batch_dim(t) for t in (q, k, v))
        probs = attn.get_attention_scores(q, k, None)      # softmax over scores rounded to q.dtype (:157)
        o = attn.batch_to_head_dim(torch.bmm(probs, v))   # (:158-159)
        y = attn.to_out[0](o) + s * self.to_out_lora(o)
        y = attn.to_out[1](y)
        return _finish(attn, y, residual, shape4)


class ConsistentIPAttnRef(nn.Module):
    def __init__(self, hidden_size, cross_attention_dim=None, rank=4, network_alpha=None, lora_scale=1.0,
                 scale=1.0, num_tokens=4):
        super().__init__()
        self.rank, self.lora_scale, self.num_tokens = rank, lora_scale, num_tokens
        self.hidden_size, self.cross_attention_dim, self.scale = hidden_size, cross_attention_dim, scale
        kv_in = cross_attention_dim or hidden_size
        self.to_q_lora = LoRALinearRef(hidden_size, hidden_size, rank, network_alpha)
        self.to_k_lora = LoRALinearRef(kv_in, hidden_size, rank, network_alpha)
        self.to_v_lora = LoRALinearRef(kv_in, hidden_size, rank, network_alpha)
        self.to_out_lora = LoRALinearRef(hidden_size, hidden_size, rank, network_alpha)
        self.to_k_ip = nn.Linear(kv_in, hidden_size, bias=False)
        self.to_v_ip = nn.Linear(kv_in, hidden_size, bias=False)

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, scale=1.0, temb=None):
        residual = hidden_states
        x, shape4 = _flatten_spatial(hidden_states)
        b = x.shape[0]
        s = self.lora_scale
        q = attn.to_q(x) + s * self.to_q_lora(x)
        if encoder_hidden_states is None:
            text, ip = x, None
        else:
            cut = encoder_hidden_states.shape[1] - self.num_tokens           # (:241-245)
            text, ip = encoder_hidden_states[:, :cut], encoder_hidden_states[:, cut:]
        k = attn.to_k(text) + s * self.to_k_lora(text)
        v = attn.to_v(text) + s * self.to_v_lora(text)
        h = attn.heads
        d = k.shape[-1] // h

        def heads_first(t):
            return t.view(b, -1, h, d).transpose(1, 2)

        qh = heads_first(q)
        o = F.scaled_dot_product_attention(qh, heads_first(k), heads_first(v), attn_mask=None, dropout_p=0.0)
        o = o.transpose(1, 2).reshape(b, -1, h * d).to(q.dtype)
        k_ip, v_ip = self.to_k_ip(ip), self.to_v_ip(ip)                       # (:266-267) no LoRA here
        o_ip = F.scaled_dot_product_attention(qh, heads_first(k_ip), heads_first(v_ip), attn_mask=None, dropout_p=0.0)
        o_ip = o_ip.transpose(1, 2).reshape(b, -1, h * d).to(q.dtype)
        o = o + self.scale * o_ip                                             # (:279)
        y = attn.to_out[0](o) + s * self.to_out_lora(o)
        y = attn.to_out[1](y)
        return _finish(attn, y, residual, shape4)


def install_ref_processors(unet, rank=128, num_tokens=4, cls_self=ConsistentAttnRef, cls_cross=ConsistentIPAttnRef):
    """``set_ip_adapter`` (pipline_StableDiffusion_ConsistentID.py:152-174)."""
    cfg = unet.config
    procs = {}
    for name in unet.attn_processors.keys():
        cad = None if name.endswith("attn1.processor") else cfg.cross_attention_dim
        if name.startswith("mid_block"):
            hidden = cfg.block_out_channels[-1]
        elif name.startswith("up_blocks"):
            hidden = list(reversed(cfg.block_out_channels))[int(name[len("up_blocks.")])]
        else:
            hidden = cfg.block_out_channels[int(name[len("down_blocks.")])]
        if cad is None:
            procs[name] = cls_self(hidden_size=hidden, cross_attention_dim=None, rank=rank)
        else:
            procs[name] = cls_cross(hidden_size=hidden, cross_attention_dim=cad, scale=1.0, rank=rank,
                                    num_tokens=num_tokens)
    unet.set_attn_processor(procs)
    return procs
