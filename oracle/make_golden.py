"""Generate tests/golden/processors/ (safetensors shards, oracle/golden.py) by EXECUTING THE REFERENCE'S OWN CODE
(unmodified adapter/attention_processor.py and adapter/resampler.py of the reference source tree) in fp32 on seeded inputs:
    python oracle/make_golden.py <reference source tree>
The reference file needs two diffusers symbols (attention_processor.py:6-7); oracle/_shim supplies them. The `attn`
argument is oracle.unet.Attention (the diffusers-0.24 Attention surface the processors touch: to_q/to_k/to_v/
to_out/heads/spatial_norm/group_norm/norm_cross/residual_connection/rescale_output_factor/prepare_attention_mask).

All inputs and weights are rounded to bf16-representable values before the fp32 reference run, so the bf16 CUDA
path consumes bit-identical operands and the only difference is arithmetic precision.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "_shim"))
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REF)

import importlib.util  # noqa: E402


def _load_reference(name, path):
    """The reference's `adapter/` has no __init__.py (a namespace package), so this repo's `adapter` package of the same name
    would shadow it on any sys.path order: load the reference FILES by path."""
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


ref_ap = _load_reference("reference_attention_processor", os.path.join(REF, "adapter", "attention_processor.py"))
ref_rs = _load_reference("reference_resampler", os.path.join(REF, "adapter", "resampler.py"))

from oracle.unet import Attention  # noqa: E402

assert ref_ap.__file__.startswith(REF), ref_ap.__file__

G = torch.Generator().manual_seed(1234)


def q(t):
    """round to bf16-representable fp32"""
    return t.bfloat16().float()


def rnd(*shape, scale=1.0):
    return q(torch.randn(*shape, generator=G) * scale)


def fill_(module, scale=None):
    with torch.no_grad():
        for n, p in module.named_parameters():
            if p.dim() >= 2:
                s = scale if scale is not None else p.shape[-1] ** -0.5
                p.copy_(rnd(*p.shape, scale=s))
            elif "norm" in n and n.endswith("weight"):
                p.copy_(q(1 + 0.1 * torch.randn(p.shape, generator=G)))
            else:
                p.copy_(rnd(*p.shape, scale=0.05))


out = {}


def put(prefix, module=None, **tensors):
    if module is not None:
        for n, p in module.state_dict().items():
            out[f"{prefix}.w.{n}"] = p.detach().clone().bfloat16()
    for k, v in tensors.items():
        out[f"{prefix}.{k}"] = v.detach().clone().contiguous()


torch.set_grad_enabled(False)
C, H, B, L, LREF, NAME = 160, 4, 2, 96, 128, "down_blocks.0.attentions.0.transformer_blocks.0.attn1.processor"

# ---- RefSAttnProcessor2_0 (hybrid self + garment attention), with and without sa_hidden_states
attn = Attention(C, None, H)
fill_(attn)
proc = ref_ap.RefSAttnProcessor2_0(NAME, C, scale=0.9)
fill_(proc)
x, g = rnd(B, L, C), rnd(B, LREF, C)
put("refs", attn, x=x.bfloat16(), g=g.bfloat16(), out=proc(attn, x, sa_hidden_states={NAME: g}), out_nosa=proc(attn, x))
put("refs.proc", proc)

# ---- CacheAttnProcessor2_0 (garment UNet tap)
cache = ref_ap.CacheAttnProcessor2_0()
y = cache(attn, x)
assert torch.equal(cache.cache["hidden_states"], x)
put("cache", out=y)

# ---- CAttnProcessor2_0 (text cross-attention, 77 tokens x 256-d here; 768-d in production)
attn2 = Attention(C, 256, H)
fill_(attn2)
cproc = ref_ap.CAttnProcessor2_0(NAME.replace("attn1", "attn2"), C, 256)
t = rnd(B, 77, 256)
put("cattn", attn2, x=x.bfloat16(), t=t.bfloat16(), out=cproc(attn2, x, encoder_hidden_states=t, sa_hidden_states={NAME: g}))

# ---- LoraRefSAttnProcessor2_0 (rank 16 here; reference uses 128)
lproc = ref_ap.LoraRefSAttnProcessor2_0(NAME, C, scale=0.8, rank=16, lora_scale=0.2)
fill_(lproc)
put("lorarefs.proc", lproc)
put("lorarefs", out=lproc(attn, x, sa_hidden_states={NAME: g}))

# ---- RefLoraSAttnProcessor2_0 (app.py variant; same arithmetic)
rlproc = ref_ap.RefLoraSAttnProcessor2_0(NAME, C, scale=0.8, rank=16, lora_scale=0.2)
rlproc.load_state_dict(lproc.state_dict())
put("reflora", out=rlproc(attn, x, sa_hidden_states={NAME: g}))

# ---- LoRAIPAttnProcessor2_0 (77 text + 4 IP tokens)
ipproc = ref_ap.LoRAIPAttnProcessor2_0(C, 256, rank=16, lora_scale=0.2, scale=0.9, num_tokens=4)
fill_(ipproc)
t81 = rnd(B, 81, 256)
put("loraip.proc", ipproc)
put("loraip", t=t81.bfloat16(), out=ipproc(attn2, x, encoder_hidden_states=t81),
    out_noface=ipproc(attn2, x, encoder_hidden_states=t))  # B11: last 4 text tokens routed to the IP stream

# ---- Resampler / ProjPlusModel (small dims; same code path as the 768-d production config)
rs = ref_rs.Resampler(dim=128, depth=2, dim_head=64, heads=2, num_queries=16, embedding_dim=256, output_dim=128, ff_mult=4)
fill_(rs)
with torch.no_grad():
    rs.latents.copy_(q(rs.latents))
clip = rnd(B, 257, 256)
put("resampler", rs, x=clip.bfloat16(), out=rs(clip))
pp = ref_rs.ProjPlusModel(cross_attention_dim=128, id_embeddings_dim=64, clip_embeddings_dim=256, num_tokens=4)
fill_(pp)
idemb = rnd(B, 64)
put("projplus", pp, id=idemb.bfloat16(), clip=clip.bfloat16(), out=pp(idemb, clip, shortcut=False),
    out_shortcut=pp(idemb, clip, shortcut=True, scale=0.5))

# ---- (appended in round 2, AFTER everything above so the seeded values of the earlier goldens do not move)
# SAttnProcessor2_0: concat-KV single softmax (:155-161); RefCAttnProcessor2_0: cross-attention + reference branch (:630-744)
sproc = ref_ap.SAttnProcessor2_0(NAME, C)
put("sattn", out=sproc(attn, x, sa_hidden_states={NAME: rnd(B, LREF, C)}), out_nosa=sproc(attn, x))
g2 = rnd(B, LREF, C)
put("sattn", g=g2.bfloat16(), out_g=sproc(attn, x, sa_hidden_states={NAME: g2}))
rcproc = ref_ap.RefCAttnProcessor2_0(NAME.replace("attn1", "attn2"), C, 256, scale=0.7)
fill_(rcproc)
NAME2 = NAME.replace("attn1", "attn2")
put("refc.proc", rcproc)
put("refc", out=rcproc(attn2, x, encoder_hidden_states=t, sa_hidden_states={NAME2: g2}),
    out_nosa=rcproc(attn2, x, encoder_hidden_states=t))

from oracle import golden  # noqa: E402

n = golden.save_processors(out, metadata={"generator": "oracle/make_golden.py", "torch": torch.__version__})
print(f"wrote {golden.PROCESSORS}: {len(out)} tensors in {n} shards")
