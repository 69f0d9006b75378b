"""CPU / eager reference of the CLIP text encoder: ``text_encoder(ids)`` / ``text_encoder_2(ids, output_hidden_states=True)``
(pipline_StableDiffusion_ConsistentID.py:467-475, pipline_StableDiffusionXL_ConsistentID.py:514-521; transformers ``CLIPTextModel`` /
``CLIPTextModelWithProjection``, state_dict keys ``text_model.*`` and ``text_projection.weight``).

TEST INFRASTRUCTURE ONLY, like oracle/: the product never imports it.  It reuses the LayerNorm / Linear helpers of oracle/clip_ref.py and
restates the encoder layer with the text transformer's causal mask.  PINNED: tests/test_clip_text_cpu.py checks it against the installed
transformers on random weights (every hidden state, last_hidden_state, pooler_output, text_embeds).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.clip_ref import _lin, _ln


def causal_encoder_layer(sd, p, x, heads, act="quick_gelu", eps=1e-5):
    """One pre-LN CLIP encoder layer in which query i attends to keys 0..i."""
    b, n, c = x.shape
    d = c // heads
    h = _ln(sd, p + ".layer_norm1", x, eps)
    split = lambda t: t.reshape(b, n, heads, d).transpose(1, 2)
    q, k, v = split(_lin(sd, p + ".self_attn.q_proj", h)), split(_lin(sd, p + ".self_attn.k_proj", h)), split(_lin(sd, p + ".self_attn.v_proj", h))
    s = ((q * d ** -0.5) @ k.transpose(-1, -2)).masked_fill(torch.ones(n, n, dtype=torch.bool, device=x.device).triu(1), float("-inf"))
    x = x + _lin(sd, p + ".self_attn.out_proj", (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(b, n, c))
    h = _lin(sd, p + ".mlp.fc1", _ln(sd, p + ".layer_norm2", x, eps))
    h = F.gelu(h) if act == "gelu" else h * torch.sigmoid(1.702 * h)      # "quick_gelu" of the OpenAI checkpoints
    return x + _lin(sd, p + ".mlp.fc2", h)


def text_hidden_states(sd, ids, heads, act="quick_gelu", eos_token_id=2, eps=1e-5):
    """-> (hidden_states, last_hidden_state, pooler_output, text_embeds or None).
    hidden_states[0] = token + position embeddings (no pre-LN), hidden_states[i] = output of layer i;
    last_hidden_state = final_layer_norm(hidden_states[-1]); the pooled row is at argmax(ids) for the legacy eos_token_id == 2, else at the
    first ids == eos_token_id; text_embeds = text_projection(pooled) (no bias) when the state dict has one."""
    n_layers = 1 + max(int(k.split(".")[3]) for k in sd if k.startswith("text_model.encoder.layers."))
    tok, pos = sd["text_model.embeddings.token_embedding.weight"], sd["text_model.embeddings.position_embedding.weight"]
    ids = ids.to(tok.device)
    hs = [tok[ids] + pos[:ids.shape[1]][None]]
    for i in range(n_layers):
        hs.append(causal_encoder_layer(sd, f"text_model.encoder.layers.{i}", hs[-1], heads, act, eps))
    last = _ln(sd, "text_model.final_layer_norm", hs[-1], eps)
    row = ids.argmax(-1) if eos_token_id == 2 else (ids == eos_token_id).int().argmax(-1)
    pooled = last[torch.arange(ids.shape[0], device=ids.device), row]
    proj = sd.get("text_projection.weight")
    return hs, last, pooled, None if proj is None else pooled @ proj.T
