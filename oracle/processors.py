"""Oracle restatement of the reference's attention processors and Perceiver resampler. TEST INFRASTRUCTURE ONLY.

Each function follows the cited lines of /root/reference/adapter/attention_processor.py and adapter/resampler.py.
PINNED: tests/test_oracle_golden.py checks these against tests/golden/processors/, produced by
oracle/make_golden.py from the reference's own classes executed (unmodified) in the build container.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


def _heads(t: torch.Tensor, B: int, h: int) -> torch.Tensor:
    return t.view(B, -1, h, t.shape[-1] // h).transpose(1, 2)


def _sdpa(q, k, v, B, h):
    """F.scaled_dot_product_attention with default 1/sqrt(d) scale, no mask (attention_processor.py:589-591)."""
    o = F.scaled_dot_product_attention(_heads(q, B, h), _heads(k, B, h), _heads(v, B, h))
    return o.transpose(1, 2).reshape(B, -1, q.shape[-1])


class CacheAttnProcessor:
    """CacheAttnProcessor2_0 (attention_processor.py:13-100): stash the processor input, then plain SDPA."""

    def __init__(self):
        self.cache: Dict[str, torch.Tensor] = {}

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, **kw):
        self.cache["hidden_states"] = hidden_states  # :34
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        B = hidden_states.shape[0]
        o = _sdpa(attn.to_q(hidden_states), attn.to_k(ctx), attn.to_v(ctx), B, attn.heads)
        return attn.to_out[1](attn.to_out[0](o))


class RefSAttnProcessor(nn.Module):
    """RefSAttnProcessor2_0 (attention_processor.py:513-627): self SDPA + scale * SDPA(q, to_k_ref(g), to_v_ref(g))."""

    def __init__(self, name, hidden_size, cross_attention_dim=None, scale=1.0):
        super().__init__()
        self.name = name
        self.to_k_ref = nn.Linear(cross_attention_dim or hidden_size, hidden_size, bias=False)  # :527
        self.to_v_ref = nn.Linear(cross_attention_dim or hidden_size, hidden_size, bias=False)  # :528
        self.scale = scale

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0,
                 num_images_per_prompt=1, cond_hidden_states=None, sa_hidden_states=None):
        B = hidden_states.shape[0]
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        q = attn.to_q(hidden_states)  # :568
        o = _sdpa(q, attn.to_k(ctx), attn.to_v(ctx), B, attn.heads)  # :575-594
        if sa_hidden_states is not None:  # :597
            g = sa_hidden_states[self.name]  # :598
            o = o + _sdpa(q, self.to_k_ref(g), self.to_v_ref(g), B, attn.heads) * self.scale  # :600-612
        return attn.to_out[1](attn.to_out[0](o))  # :615-617


class CAttnProcessor(nn.Module):
    """CAttnProcessor2_0 (attention_processor.py:202-295): plain (text) cross-attention; ignores sa_hidden_states."""

    def __init__(self, name=None, hidden_size=None, cross_attention_dim=None):
        super().__init__()
        self.name = name

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, **kw):
        B = hidden_states.shape[0]
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        o = _sdpa(attn.to_q(hidden_states), attn.to_k(ctx), attn.to_v(ctx), B, attn.heads)
        return attn.to_out[1](attn.to_out[0](o))


class SAttnProcessor(nn.Module):
    """SAttnProcessor2_0 (attention_processor.py:103-200): ONE softmax over the concatenated keys — for self-attention with
    garment features the context is cat([hidden_states, sa_hidden_states[name]], dim=1) (:155-161), projected by the layer's
    own to_k / to_v."""

    def __init__(self, name, hidden_size=None, cross_attention_dim=None):
        super().__init__()
        self.name = name

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0,
                 cond_hidden_states=None, sa_hidden_states=None):
        B = hidden_states.shape[0]
        if encoder_hidden_states is None:
            ctx = hidden_states if sa_hidden_states is None else torch.cat([hidden_states, sa_hidden_states[self.name]], 1)
        else:
            ctx = encoder_hidden_states
        o = _sdpa(attn.to_q(hidden_states), attn.to_k(ctx), attn.to_v(ctx), B, attn.heads)  # :163-182
        return attn.to_out[1](attn.to_out[0](o))


class RefCAttnProcessor(nn.Module):
    """RefCAttnProcessor2_0 (attention_processor.py:630-744): (cross-)attention + scale * SDPA(q, to_k_ref(g), to_v_ref(g));
    to_k_ref / to_v_ref take hidden_size inputs (:643-644)."""

    def __init__(self, name, hidden_size, cross_attention_dim=None, scale=1.0):
        super().__init__()
        self.name = name
        self.to_k_ref = nn.Linear(hidden_size, hidden_size, bias=False)
        self.to_v_ref = nn.Linear(hidden_size, hidden_size, bias=False)
        self.scale = scale

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0,
                 cond_hidden_states=None, sa_hidden_states=None):
        B = hidden_states.shape[0]
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        q = attn.to_q(hidden_states)
        o = _sdpa(q, attn.to_k(ctx), attn.to_v(ctx), B, attn.heads)  # :691-706
        if sa_hidden_states is not None:  # :709-727
            g = sa_hidden_states[self.name]
            o = o + _sdpa(q, self.to_k_ref(g), self.to_v_ref(g), B, attn.heads) * self.scale
        return attn.to_out[1](attn.to_out[0](o))


class LoRALinear(nn.Module):
    """diffusers-0.24 LoRALinearLayer with network_alpha=None: up(down(x)) (SURVEY.md A.5)."""

    def __init__(self, cin, cout, rank):
        super().__init__()
        self.down = nn.Linear(cin, rank, bias=False)
        self.up = nn.Linear(rank, cout, bias=False)

    def forward(self, x):
        return self.up(self.down(x))


class LoraRefSAttnProcessor(nn.Module):
    """LoraRefSAttnProcessor2_0 (attention_processor.py:391-511): RefS + lora_scale * LoRA on q, k, v, out."""

    def __init__(self, name, hidden_size, cross_attention_dim=None, rank=4, lora_scale=1.0, scale=1.0):
        super().__init__()
        self.name, self.scale, self.lora_scale = name, scale, lora_scale
        kv = cross_attention_dim or hidden_size
        self.to_q_lora = LoRALinear(hidden_size, hidden_size, rank)
        self.to_k_lora = LoRALinear(kv, hidden_size, rank)
        self.to_v_lora = LoRALinear(kv, hidden_size, rank)
        self.to_out_lora = LoRALinear(hidden_size, hidden_size, rank)
        self.to_k_ref = nn.Linear(kv, hidden_size, bias=False)
        self.to_v_ref = nn.Linear(kv, hidden_size, bias=False)

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0,
                 sa_hidden_states=None, **kw):
        B = hidden_states.shape[0]
        ls = self.lora_scale
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        q = attn.to_q(hidden_states) + ls * self.to_q_lora(hidden_states)  # :453
        k = attn.to_k(ctx) + ls * self.to_k_lora(ctx)  # :461
        v = attn.to_v(ctx) + ls * self.to_v_lora(ctx)  # :462
        o = _sdpa(q, k, v, B, attn.heads)
        if sa_hidden_states is not None:
            g = sa_hidden_states[self.name]
            o = o + _sdpa(q, self.to_k_ref(g), self.to_v_ref(g), B, attn.heads) * self.scale
        o = attn.to_out[0](o) + ls * self.to_out_lora(o)  # :500
        return attn.to_out[1](o)


class LoRAIPAttnProcessor(nn.Module):
    """LoRAIPAttnProcessor2_0 (attention_processor.py:746-871): text SDPA (LoRA q/k/v) + scale * SDPA over the last
    num_tokens context tokens through to_k_ip / to_v_ip; out projection + LoRA."""

    def __init__(self, hidden_size, cross_attention_dim=None, rank=4, lora_scale=1.0, scale=1.0, num_tokens=4):
        super().__init__()
        self.lora_scale, self.scale, self.num_tokens = lora_scale, scale, num_tokens
        kv = cross_attention_dim or hidden_size
        self.to_q_lora = LoRALinear(hidden_size, hidden_size, rank)
        self.to_k_lora = LoRALinear(kv, hidden_size, rank)
        self.to_v_lora = LoRALinear(kv, hidden_size, rank)
        self.to_out_lora = LoRALinear(hidden_size, hidden_size, rank)
        self.to_k_ip = nn.Linear(kv, hidden_size, bias=False)
        self.to_v_ip = nn.Linear(kv, hidden_size, bias=False)

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, scale=1.0, temb=None,
                 *args, **kw):
        B = hidden_states.shape[0]
        ls = self.lora_scale
        q = attn.to_q(hidden_states) + ls * self.to_q_lora(hidden_states)  # :804
        end = encoder_hidden_states.shape[1] - self.num_tokens  # :811
        text, ip = encoder_hidden_states[:, :end], encoder_hidden_states[:, end:]  # :812-815
        k = attn.to_k(text) + ls * self.to_k_lora(text)  # :820
        v = attn.to_v(text) + ls * self.to_v_lora(text)  # :821
        o = _sdpa(q, k, v, B, attn.heads)  # :833
        o = o + self.scale * _sdpa(q, self.to_k_ip(ip), self.to_v_ip(ip), B, attn.heads)  # :841-856
        o = attn.to_out[0](o) + ls * self.to_out_lora(o)  # :859
        return attn.to_out[1](o)


# ------------------------------------------------------------------ adapter/resampler.py
class PerceiverAttention(nn.Module):
    """adapter/resampler.py:34-78."""

    def __init__(self, dim, dim_head=64, heads=8):
        super().__init__()
        self.dim_head, self.heads = dim_head, heads
        inner = dim_head * heads
        self.norm1, self.norm2 = nn.LayerNorm(dim), nn.LayerNorm(dim)
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_kv = nn.Linear(dim, inner * 2, bias=False)
        self.to_out = nn.Linear(inner, dim, bias=False)

    def forward(self, x, latents):
        x, latents = self.norm1(x), self.norm2(latents)  # :57-58
        b, l, _ = latents.shape
        q = self.to_q(latents)
        k, v = self.to_kv(torch.cat((x, latents), dim=-2)).chunk(2, dim=-1)  # :63-64
        q, k, v = (_heads(t, b, self.heads) for t in (q, k, v))
        s = 1 / math.sqrt(math.sqrt(self.dim_head))  # :71
        w = torch.softmax(((q * s) @ (k * s).transpose(-2, -1)).float(), dim=-1).type(q.dtype)  # :72-73
        out = (w @ v).permute(0, 2, 1, 3).reshape(b, l, -1)
        return self.to_out(out)


def _ff(dim, mult=4):
    """adapter/resampler.py:13-20."""
    return nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, dim * mult, bias=False), nn.GELU(),
                         nn.Linear(dim * mult, dim, bias=False))


class Resampler(nn.Module):
    """adapter/resampler.py:170-236 with apply_pos_emb=False, num_latents_mean_pooled=0 (the reference's use,
    inference_IMAGdressing.py:55-65)."""

    def __init__(self, dim=1024, depth=8, dim_head=64, heads=16, num_queries=8, embedding_dim=768, output_dim=1024,
                 ff_mult=4):
        super().__init__()
        self.latents = nn.Parameter(torch.randn(1, num_queries, dim) / dim ** 0.5)
        self.proj_in = nn.Linear(embedding_dim, dim)
        self.proj_out = nn.Linear(dim, output_dim)
        self.norm_out = nn.LayerNorm(output_dim)
        self.layers = nn.ModuleList(
            [nn.ModuleList([PerceiverAttention(dim, dim_head, heads), _ff(dim, ff_mult)]) for _ in range(depth)])

    def forward(self, x):
        latents = self.latents.repeat(x.size(0), 1, 1)
        x = self.proj_in(x)
        for attn, ff in self.layers:
            latents = attn(x, latents) + latents
            latents = ff(latents) + latents
        return self.norm_out(self.proj_out(latents))


class ProjPlusModel(nn.Module):
    """adapter/resampler.py:250-281 (FacePerceiverResampler :128-167 inlined as `perceiver_resampler`)."""

    def __init__(self, cross_attention_dim=768, id_embeddings_dim=512, clip_embeddings_dim=1280, num_tokens=4):
        super().__init__()
        self.cross_attention_dim, self.num_tokens = cross_attention_dim, num_tokens
        self.proj = nn.Sequential(nn.Linear(id_embeddings_dim, id_embeddings_dim * 2), nn.GELU(),
                                  nn.Linear(id_embeddings_dim * 2, cross_attention_dim * num_tokens))
        self.norm = nn.LayerNorm(cross_attention_dim)
        d = cross_attention_dim

        class _FPR(nn.Module):
            def __init__(s):
                super().__init__()
                s.proj_in = nn.Linear(clip_embeddings_dim, d)
                s.proj_out = nn.Linear(d, d)
                s.norm_out = nn.LayerNorm(d)
                s.layers = nn.ModuleList(
                    [nn.ModuleList([PerceiverAttention(d, 64, d // 64), _ff(d, 4)]) for _ in range(4)])

            def forward(s, latents, x):
                x = s.proj_in(x)
                for attn, ff in s.layers:
                    latents = attn(x, latents) + latents
                    latents = ff(latents) + latents
                return s.norm_out(s.proj_out(latents))

        self.perceiver_resampler = _FPR()

    def forward(self, id_embeds, clip_embeds, shortcut=False, scale=1.0):
        x = self.norm(self.proj(id_embeds).reshape(-1, self.num_tokens, self.cross_attention_dim))
        out = self.perceiver_resampler(x, clip_embeds)
        return x + scale * out if shortcut else out
