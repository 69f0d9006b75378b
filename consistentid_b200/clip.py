"""CLIP ViT image encoder on the GPU (SURVEY.md 8f-4): ``image_encoder(pixels, output_hidden_states=True).hidden_states[-2]``
(pipline_StableDiffusion_ConsistentID.py:182-183, 202-203; ``laion/CLIP-ViT-H-14``: 1280 wide, 32 layers of which the last is never
needed, 16 heads of 80, 257 tokens; the pipeline pushes the face crop, the 5 facial-region crops and their zero images through it).
Takes the ``vision_model.*`` entries of a transformers ``CLIPVisionModelWithProjection`` state_dict.

Kernels reused from the hot path: ``cid_gemm`` (patch embedding as a GEMM over unfolded 14x14 patches with K 588 -> 640, fused-bias QKV
with the transposed-V epilogue, out-proj / fc2 with fused bias + residual, fc1 with the fused exact-erf GELU epilogue), ``cid_layernorm``,
``cid_attn_self_ragged`` (the 257 tokens live in 264-row buffers; the 7 pad keys are masked inside the flash kernel), ``cid_add_inplace``.
16-bit CUDA tensors only; there is no CPU / fp32 path.

B200CLIPTextEncoder: the CLIP text transformer (SD1.5 ``text_encoder`` = OpenAI ViT-L/14, SDXL ``text_encoder_2`` = OpenCLIP ViT-bigG/14),
the same pre-LN layer stack with a causal mask (``cid_attn_self_causal``), QuickGELU or GELU in the fc1 epilogue, a token + position
embedding gather (``cid_embed_tokens``) in front and final LayerNorm + EOS pooling + projection behind.
"""
from __future__ import annotations

import types

import torch
import torch.nn.functional as F

from . import ops
from .lib import EPI_GELU, EPI_QKV, EPI_QUICK_GELU


def _load_layers(W, prefix, n_layers):
    """Packed weights of ``n_layers`` CLIP encoder layers (``{prefix}{i}.*`` state_dict keys): fused QKV weight / bias, out-proj, MLP, LNs."""
    p = {}
    for i in range(n_layers):
        b = f"{prefix}{i}."
        for ln in ("layer_norm1", "layer_norm2"):
            p[f"{i}.{ln}.g"], p[f"{i}.{ln}.b"] = W(b + ln + ".weight"), W(b + ln + ".bias")
        p[f"{i}.qkv.w"] = torch.cat([W(b + f"self_attn.{q}_proj.weight") for q in "qkv"], 0).contiguous()
        p[f"{i}.qkv.b"] = torch.cat([W(b + f"self_attn.{q}_proj.bias") for q in "qkv"], 0).contiguous()
        p[f"{i}.o.w"], p[f"{i}.o.b"] = W(b + "self_attn.out_proj.weight"), W(b + "self_attn.out_proj.bias")
        p[f"{i}.fc1.w"], p[f"{i}.fc1.b"] = W(b + "mlp.fc1.weight"), W(b + "mlp.fc1.bias")
        p[f"{i}.fc2.w"], p[f"{i}.fc2.b"] = W(b + "mlp.fc2.weight"), W(b + "mlp.fc2.bias")
    inter = p["0.fc1.w"].shape[0] if n_layers else None
    if inter is not None and inter % 64:
        raise ValueError(f"intermediate size {inter} must be a multiple of 64")
    return p


def _encoder_stack(p, x, n_layers, B, Np, heads, act_epi, attend, eps=1e-5, hidden_states=None):
    """The pre-LN CLIP encoder layers on x [B*Np, C] (16-bit rows, Np tokens per sample): LN1 -> QKV GEMM with the transposed-V epilogue ->
    attend(q, k, vt, out) -> out-proj + bias + residual -> LN2 -> fc1 + bias + ``act_epi`` -> fc2 + bias + residual.  Each layer writes a
    fresh output buffer; ``hidden_states`` (a list) collects them."""
    M, C = x.shape
    d = C // heads
    new = lambda *s: torch.empty(s, dtype=x.dtype, device=x.device)
    inter = p["0.fc1.w"].shape[0] if n_layers else C
    h, qk, vt, ao, mid = new(M, C), new(M, 2 * C), new(B * heads, d, Np), new(M, C), new(M, inter)
    for i in range(n_layers):
        ops.layernorm(x, p[f"{i}.layer_norm1.g"], p[f"{i}.layer_norm1.b"], h, M, C, eps)
        ops.gemm(h, p[f"{i}.qkv.w"], qk, bias=p[f"{i}.qkv.b"], epi=EPI_QKV, vt=vt, n_split=2 * C, heads=heads, hdim=d, ntok=Np)
        attend(qk[:, :C], qk[:, C:], vt, ao)
        x = ops.gemm(ao, p[f"{i}.o.w"], new(M, C), bias=p[f"{i}.o.b"], residual=x)
        ops.layernorm(x, p[f"{i}.layer_norm2.g"], p[f"{i}.layer_norm2.b"], h, M, C, eps)
        ops.gemm(h, p[f"{i}.fc1.w"], mid, bias=p[f"{i}.fc1.b"], epi=act_epi)
        x = ops.gemm(mid, p[f"{i}.fc2.w"], new(M, C), bias=p[f"{i}.fc2.b"], residual=x)
        if hidden_states is not None:
            hidden_states.append(x)
    return x


class B200CLIPVisionEncoder:
    def __init__(self, state_dict, num_attention_heads=16, hidden_act="gelu", dtype=torch.float16, device="cuda"):
        if hidden_act != "gelu":
            raise NotImplementedError("only hidden_act='gelu' (the laion ViT-H/14 the reference loads) is implemented")
        self.dtype, self.device, self.heads = dtype, torch.device(device), num_attention_heads
        ops.ensure_workspace(self.device)
        W = lambda n: state_dict[n].detach().to(device=self.device, dtype=dtype).contiguous()
        pw = W("vision_model.embeddings.patch_embedding.weight")                    # [C, 3, P, P]
        self.C, self.P = pw.shape[0], pw.shape[-1]
        if self.C % 64 or (self.C // num_attention_heads) % 8:
            raise ValueError(f"hidden size {self.C} / heads {num_attention_heads}: need C % 64 == 0 and head dim % 8 == 0")
        k = 3 * self.P * self.P
        self.Kp = (k + 63) // 64 * 64
        wp = torch.zeros((self.C, self.Kp), dtype=dtype, device=self.device)
        wp[:, :k] = pw.reshape(self.C, k)
        self.p = p = {"patch.w": wp, "cls": W("vision_model.embeddings.class_embedding"), "pos": W("vision_model.embeddings.position_embedding.weight")}
        self.n_tok = p["pos"].shape[0]
        self.n_pad = (self.n_tok + 7) // 8 * 8
        n_layers = 1 + max(int(n.split(".")[3]) for n in state_dict if n.startswith("vision_model.encoder.layers."))
        self.n_run = n_layers - 1                                                         # hidden_states[-2]: the last layer is skipped
        p["pre_layrnorm.g"], p["pre_layrnorm.b"] = W("vision_model.pre_layrnorm.weight"), W("vision_model.pre_layrnorm.bias")
        p.update(_load_layers(W, "vision_model.encoder.layers.", self.n_run))

    @torch.no_grad()
    def __call__(self, pixel_values):
        """pixel_values [B, 3, H, W] (H, W multiples of the patch size) -> hidden_states[-2] [B, 1 + n_patches, C]."""
        if not (pixel_values.is_cuda and pixel_values.dtype == self.dtype and pixel_values.ndim == 4):
            raise TypeError(f"B200CLIPVisionEncoder: expected a CUDA {self.dtype} tensor [B, 3, H, W] (no CPU/fp32 path)")
        p, C, H, Np = self.p, self.C, self.heads, self.n_pad
        d = C // H
        B = pixel_values.shape[0]
        new = lambda *s: torch.empty(s, dtype=self.dtype, device=self.device)
        cols = F.unfold(pixel_values, kernel_size=self.P, stride=self.P).transpose(1, 2)          # [B, n_patches, 3*P*P] (data movement only)
        n_patch = cols.shape[1]
        if n_patch + 1 != self.n_tok:
            raise ValueError(f"{n_patch} patches + class token != {self.n_tok} position embeddings")
        a = torch.zeros((B * n_patch, self.Kp), dtype=self.dtype, device=self.device)
        a[:, :cols.shape[2]] = cols.reshape(B * n_patch, -1)
        patches = ops.gemm(a, p["patch.w"], new(B * n_patch, C))
        x = torch.zeros((B, Np, C), dtype=self.dtype, device=self.device)
        x[:, 0] = p["cls"]
        x[:, 1:self.n_tok] = patches.view(B, n_patch, C)
        pos = torch.zeros((B, Np, C), dtype=self.dtype, device=self.device)
        pos[:, :self.n_tok] = p["pos"]
        ops.add_inplace(x, pos)
        M = B * Np
        x = ops.layernorm(x.view(M, C), p["pre_layrnorm.g"], p["pre_layrnorm.b"], new(M, C), M, C)
        attend = lambda q, k, vt, out: ops.attn_self(q, k, vt, out, B, H, Np, d, n_valid=self.n_tok)
        x = _encoder_stack(p, x, self.n_run, B, Np, H, EPI_GELU, attend)
        return x.view(B, Np, C)[:, :self.n_tok].contiguous()


class CLIPTextOutput:
    """The fields of transformers' ``BaseModelOutputWithPooling`` / ``CLIPTextModelOutput`` the pipelines read.  Indexing follows
    transformers: ``[0]`` is ``text_embeds`` for the projection variant and ``last_hidden_state`` otherwise; ``None`` fields are skipped."""

    def __init__(self, last_hidden_state, pooler_output, hidden_states=None, text_embeds=None):
        self.last_hidden_state, self.pooler_output, self.hidden_states, self.text_embeds = last_hidden_state, pooler_output, hidden_states, text_embeds

    def to_tuple(self):
        if self.text_embeds is not None:
            fields = (self.text_embeds, self.last_hidden_state, self.hidden_states)
        else:
            fields = (self.last_hidden_state, self.pooler_output, self.hidden_states)
        return tuple(f for f in fields if f is not None)

    def __getitem__(self, i):
        return self.to_tuple()[i]


class B200CLIPTextEncoder:
    """Drop-in for ``pipe.text_encoder`` (transformers ``CLIPTextModel``) and ``pipe.text_encoder_2`` (``CLIPTextModelWithProjection``).

    Takes the ``text_model.*`` entries of the state_dict, plus ``text_projection.weight`` for the projection variant.  Sequences of
    L <= max_position_embeddings tokens live in Lp = ceil8(L)-row buffers: pad rows start as zeros and stay finite, and the causal mask keeps
    real rows from reading them.  ``input_ids`` may live on the host (range-checked, then copied) or on the device (no host synchronisation)."""

    def __init__(self, state_dict, num_attention_heads=12, hidden_act="quick_gelu", eos_token_id=2, layer_norm_eps=1e-5,
                 dtype=torch.float16, device="cuda"):
        if hidden_act not in ("quick_gelu", "gelu"):
            raise NotImplementedError(f"hidden_act={hidden_act!r}: only 'quick_gelu' (OpenAI ViT-L/14) and 'gelu' (OpenCLIP ViT-bigG/14)")
        self.dtype, self.device, self.heads = dtype, torch.device(device), num_attention_heads
        self.act_epi = EPI_QUICK_GELU if hidden_act == "quick_gelu" else EPI_GELU
        self.eos_token_id, self.eps = eos_token_id, layer_norm_eps
        ops.ensure_workspace(self.device)
        W = lambda n: state_dict[n].detach().to(device=self.device, dtype=dtype).contiguous()
        self.p = p = {"tok": W("text_model.embeddings.token_embedding.weight"), "pos": W("text_model.embeddings.position_embedding.weight"),
                      "final.g": W("text_model.final_layer_norm.weight"), "final.b": W("text_model.final_layer_norm.bias")}
        self.C = p["tok"].shape[1]
        self.max_len = p["pos"].shape[0]
        if self.C % 64 or (self.C // num_attention_heads) % 8:
            raise ValueError(f"hidden size {self.C} / heads {num_attention_heads}: need C % 64 == 0 and head dim % 8 == 0")
        self.n_layers = 1 + max(int(n.split(".")[3]) for n in state_dict if n.startswith("text_model.encoder.layers."))
        p.update(_load_layers(W, "text_model.encoder.layers.", self.n_layers))
        if "text_projection.weight" in state_dict:
            p["proj.w"] = W("text_projection.weight")                                   # [projection_dim, C], no bias
        self.config = types.SimpleNamespace(hidden_size=self.C, num_hidden_layers=self.n_layers, use_attention_mask=False,
                                            projection_dim=p["proj.w"].shape[0] if "proj.w" in p else None)

    @torch.no_grad()
    def __call__(self, input_ids, attention_mask=None, output_hidden_states=False):
        """input_ids [B, L] integer token ids -> CLIPTextOutput with [B, L, C] last_hidden_state (and hidden_states), [B, C] pooler_output,
        [B, projection_dim] text_embeds (projection variant)."""
        if attention_mask is not None:
            raise NotImplementedError("attention_mask: the CLIP text encoders run unmasked (config.use_attention_mask is False)")
        if input_ids.ndim != 2 or input_ids.dtype.is_floating_point or input_ids.dtype == torch.bool:
            raise TypeError(f"B200CLIPTextEncoder: expected integer token ids [B, L], got {input_ids.dtype} {tuple(input_ids.shape)}")
        p, C, H = self.p, self.C, self.heads
        B, L = input_ids.shape
        if not 0 < L <= self.max_len:
            raise ValueError(f"{L} tokens: the encoder has {self.max_len} positions")
        ids = input_ids.to(torch.int64)
        Lp = (L + 7) // 8 * 8
        M, d = B * Lp, C // H
        new = lambda *s: torch.empty(s, dtype=self.dtype, device=self.device)
        x = ops.embed_tokens(ids, p["tok"], p["pos"], new(M, C), Lp)
        hs = [x] if output_hidden_states else None
        attend = lambda q, k, vt, out: ops.attn_self_causal(q, k, vt, out, B, H, Lp, d)
        x = _encoder_stack(p, x, self.n_layers, B, Lp, H, self.act_epi, attend, self.eps, hs)
        last = ops.layernorm(x, p["final.g"], p["final.b"], new(M, C), M, C, self.eps)
        # pooled row: argmax(ids) under the legacy eos_token_id == 2, else the first EOS (index bookkeeping only)
        row = ids.argmax(-1) if self.eos_token_id == 2 else (ids == self.eos_token_id).int().argmax(-1)
        row = row.to(self.device) + Lp * torch.arange(B, device=self.device)
        pooled = last.index_select(0, row)
        text_embeds = None
        if "proj.w" in p:
            P = p["proj.w"].shape[0]
            text_embeds = ops.skinny_linear(pooled, p["proj.w"], None, new(B, P), B, P, C)
        rows = lambda t: t.view(B, Lp, C)[:, :L].contiguous()
        return CLIPTextOutput(rows(last), pooled, None if hs is None else tuple(rows(t) for t in hs), text_embeds)
