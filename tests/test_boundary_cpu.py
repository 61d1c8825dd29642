"""CPU (kernel wrappers emulated, tests/emulated_ops.py): drop-in boundary behaviour added in round 2 —

* the `null_prompt` garment-token fallback of the reference `__call__` (IMAGDressing_v1_pipeline.py:416-435),
* the ControlNet guidance window `controlnet_keep` (IMAGDressing_v1_pipeline_ipa_controlnet.py:584-590,643-649),
* the inpainting pipeline fed PIL images the way inference_IMAGdressing_controlnetinpainting.py feeds it
  (resize / normalise / binarise, IMAGDressing_v1_pipeline_controlnet_inpainting.py:301-308),
* processors registered on a FOREIGN `Attention` host module (a stock diffusers-style module without this package's
  pack cache / fused-residual handshake),
* stale-pack protection: a reference-style `ModuleList(unet.attn_processors.values()).load_state_dict(...)` and a
  changed `image_scale` between two calls must take effect.
"""
import numpy as np
import pytest
import torch
import torch.nn as nn

import emulated_ops
from oracle import processors as op
from oracle import unet as ou
from oracle.pipeline import sample_one
from test_pipelines_cpu import H, STEPS, W, build, common, eager, inputs, rel


@pytest.fixture
def emu(monkeypatch):
    emulated_ops.install(monkeypatch)
    from imagdressing_b200 import modeling

    monkeypatch.setattr(modeling, "FOLD_LN", False)
    return modeling


def base_pipe(p, rp, sched):
    from dressing_sd.pipelines.IMAGDressing_v1_pipeline import IMAGDressing_v1

    return eager(IMAGDressing_v1(vae=None, reference_unet=rp, unet=p, tokenizer=None, text_encoder=None, image_encoder=None,
                                 ImgProj=None, scheduler=sched, safety_checker=None, feature_extractor=None))


@torch.no_grad()
def test_null_prompt_branch_uses_prompt_embeddings_as_garment_tokens(emu):
    """ref_clip_image=None: the reference's second encode_prompt call receives the already-encoded prompt_embeds and
    therefore returns them unchanged — the garment UNet's text slot is the positive prompt (quirk B19)."""
    (o, ro, _), (p, rp, _), sched = build(emu)
    x = inputs(60)
    ref = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["prompt"], x["garment"], 7.5, STEPS)
    kw = common(x)
    kw.update(garment_tokens=None, null_prompt="a null prompt that is never encoded")
    out = base_pipe(p, rp, sched)(guidance_scale=7.5, ref_clip_image=None, **kw).images
    assert rel(out, ref) < 4e-2
    other = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["gtok"], x["garment"], 7.5, STEPS)
    assert rel(other, ref) > 5e-2  # the garment tokens matter, so the match above is not vacuous


@torch.no_grad()
def test_control_guidance_window(emu):
    from dressing_sd.pipelines.IMAGDressing_v1_pipeline_controlnet import IMAGDressing_v1 as PControl

    (o, ro, co), (p, rp, cp), sched = build(emu)
    x = inputs(61)
    pipe = eager(PControl(vae=None, reference_unet=rp, unet=p, tokenizer=None, text_encoder=None, controlnet=cp,
                          image_encoder=None, ImgProj=None, scheduler=sched, safety_checker=None, feature_extractor=None))
    full = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["gtok"], x["garment"], 7.0, STEPS, controlnet=co,
                      control_cond=x["pose"], control_scale=0.8)
    win = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["gtok"], x["garment"], 7.0, STEPS, controlnet=co,
                     control_cond=x["pose"], control_scale=0.8, control_guidance_start=0.25, control_guidance_end=0.75)
    assert rel(win, full) > 1e-2
    out = pipe(guidance_scale=7.0, pose_image=x["pose"], controlnet_conditioning_scale=0.8, control_guidance_start=0.25,
               control_guidance_end=[0.75], **common(x)).images
    assert rel(out, win) < 4e-2 and rel(out, win) < rel(out, full)
    with pytest.raises(NotImplementedError):
        pipe(guidance_scale=7.0, pose_image=x["pose"], guess_mode=True, **common(x))
    with pytest.raises(ValueError):
        pipe(guidance_scale=7.0, pose_image=x["pose"], control_guidance_start=0.9, control_guidance_end=0.1, **common(x))


class ToyVAE(nn.Module):
    """8x average-pool 'VAE' stand-in (test infrastructure): encode -> latent_dist with mean / sample, 4 channels."""

    class _Dist:
        def __init__(self, mean):
            self.mean = mean

        def sample(self, generator=None):
            return self.mean

    class _Out:
        def __init__(self, d):
            self.latent_dist = d

    def __init__(self):
        super().__init__()
        self.w = nn.Parameter(torch.tensor([[1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0], [0.3, 0.3, 0.4]]))
        self.config = ou.Config(scaling_factor=0.18215, block_out_channels=(1, 1, 1, 1), latent_channels=4)

    @property
    def dtype(self):
        return self.w.dtype

    @property
    def device(self):
        return self.w.device

    def encode(self, x):
        pooled = torch.nn.functional.avg_pool2d(x.float(), 8)
        return self._Out(self._Dist(torch.einsum("oc,nchw->nohw", self.w, pooled)))


@torch.no_grad()
def test_inpainting_accepts_pil_images_like_the_reference_script(emu):
    from PIL import Image

    from dressing_sd.pipelines.IMAGDressing_v1_pipeline_controlnet_inpainting import IMAGDressing_v1 as PInpaint

    (o, ro, co), (p, rp, cp), sched = build(emu)
    vae = ToyVAE()
    pin = eager(PInpaint(vae=vae, reference_unet=rp, unet=p, tokenizer=None, text_encoder=None, controlnet=cp,
                         image_encoder=None, ImgProj=None, scheduler=sched, safety_checker=None, feature_extractor=None))
    x = inputs(62)
    rng = np.random.default_rng(0)
    # the script passes PIL images of ANOTHER size than (height, width): they must be resized, normalised, binarised
    small = (H * 8 // 2, W * 8 // 2)
    image = Image.fromarray(rng.integers(0, 255, (*small, 3), dtype=np.uint8))
    mask_np = np.zeros(small, dtype=np.uint8)
    mask_np[small[0] // 4: 3 * small[0] // 4, small[1] // 4: 3 * small[1] // 4] = 200  # grey level 200 -> 1 after binarise
    mask = Image.fromarray(mask_np)
    pose = Image.fromarray(rng.integers(0, 255, (*small, 3), dtype=np.uint8))
    kw = common(x)
    out = pin(guidance_scale=5.0, image=image, mask_image=mask, control_image=pose, strength=1.0,
              controlnet_conditioning_scale=0.5, **kw).images
    # the same call with the preprocessing done by hand, fed as tensors
    img_t = torch.from_numpy(np.asarray(image.resize((W * 8, H * 8), resample=Image.LANCZOS)).astype("float32") / 255.0)
    img_t = img_t.permute(2, 0, 1)[None] * 2 - 1
    img_lat = vae.encode(img_t).latent_dist.mean * 0.18215
    m = torch.from_numpy(np.asarray(mask.resize((W * 8, H * 8), resample=Image.LANCZOS)).astype("float32") / 255.0)
    m_lat = torch.nn.functional.interpolate((m >= 0.5).float()[None, None], size=(H, W))
    assert 0 < m_lat.sum() < m_lat.numel() and set(m_lat.unique().tolist()) == {0.0, 1.0}
    pose_t = torch.from_numpy(np.asarray(pose.resize((W * 8, H * 8), resample=Image.LANCZOS)).astype("float32") / 255.0)
    pose_t = pose_t.permute(2, 0, 1)[None]
    ref = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["gtok"], x["garment"], 5.0, STEPS, controlnet=co,
                     control_cond=pose_t, control_scale=0.5, mask=m_lat, image_latents=img_lat, noise=x["latents"])
    assert rel(out, ref) < 4e-2
    keep = (m_lat == 0).expand_as(out)
    assert rel(out[keep], img_lat[keep]) < 1e-5


@torch.no_grad()
def test_processors_on_a_foreign_attention_host(emu):
    """The drop-in processors registered on a module that is NOT imagdressing_b200.modeling.Attention (here the
    oracle's diffusers-style Attention: no `packed`, no `_fused_residual`, no `_ln_fold`): the pack cache lives on the
    processor and the residual is left to the host block, as diffusers does."""
    from adapter.attention_processor import CAttnProcessor2_0, LoraRefSAttnProcessor2_0, RefSAttnProcessor2_0

    torch.manual_seed(0)
    C, heads, L = 64, 8, 48
    host = ou.Attention(C, None, heads)
    xhost = ou.Attention(C, 32, heads)
    x, g, t = torch.randn(2, L, C), torch.randn(2, L, C), torch.randn(2, 7, 32)
    name = "down_blocks.0.attentions.0.transformer_blocks.0.attn1.processor"
    for ours, theirs in ((RefSAttnProcessor2_0(name, C, scale=0.7), op.RefSAttnProcessor(name, C, scale=0.7)),
                         (LoraRefSAttnProcessor2_0(name, C, rank=4, scale=0.7, lora_scale=0.5),
                          op.LoraRefSAttnProcessor(name, C, rank=4, lora_scale=0.5, scale=0.7))):
        for prm in ours.parameters():
            nn.init.normal_(prm, std=0.1)
        theirs.load_state_dict(ours.state_dict())
        ref = theirs(host, x, sa_hidden_states={name: g})
        out = ours(host, x, sa_hidden_states={name: g})
        assert rel(out, ref) < 2e-2
        assert not hasattr(host, "_pk") and id(host) in ours._foreign_pk
        # in-place weight edit on the host after a forward: the pack must follow (no stale copy)
        with torch.no_grad():
            host.to_q.weight.mul_(0.5)
        assert rel(ours(host, x, sa_hidden_states={name: g}), theirs(host, x, sa_hidden_states={name: g})) < 2e-2
    ours, theirs = CAttnProcessor2_0(name, C, 32), op.CAttnProcessor(name)
    assert rel(ours(xhost, x, encoder_hidden_states=t), theirs(xhost, x, encoder_hidden_states=t)) < 2e-2


@torch.no_grad()
def test_scale_change_and_processor_reload_between_calls(emu):
    (o, ro, _), (p, rp, _), sched = build(emu)
    pipe = base_pipe(p, rp, sched)
    x = inputs(63)
    a = pipe(guidance_scale=7.5, image_scale=1.0, **common(x)).images
    b = pipe(guidance_scale=7.5, image_scale=0.3, **common(x)).images
    for proc in o.attn_processors.values():
        if hasattr(proc, "scale"):
            proc.scale = 0.3
    ref_b = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["gtok"], x["garment"], 7.5, STEPS)
    assert rel(b, ref_b) < 4e-2 and rel(a, ref_b) > rel(b, ref_b)
    # reference-style adapter reload (inference_IMAGdressing.py:112-114): ModuleList over the processors
    layers_p = nn.ModuleList([v for v in p.attn_processors.values() if isinstance(v, nn.Module)])
    layers_o = nn.ModuleList([v for v in o.attn_processors.values() if isinstance(v, nn.Module)])
    sd = {k: torch.randn_like(v) * 0.05 for k, v in layers_p.state_dict().items()}
    layers_p.load_state_dict(sd)
    layers_o.load_state_dict(sd)
    c = pipe(guidance_scale=7.5, image_scale=0.3, **common(x)).images
    ref_c = sample_one(o, ro, x["latents"], x["prompt"], x["negative"], x["gtok"], x["garment"], 7.5, STEPS)
    assert rel(c, ref_c) < 4e-2 and rel(b, ref_c) > rel(c, ref_c)


@torch.no_grad()
def test_sattn_and_refc_drop_ins_match_reference_goldens(monkeypatch):
    """SAttnProcessor2_0 (concat-KV single softmax, reference :103-200) and RefCAttnProcessor2_0 (cross-attention + reference
    branch, :630-744) — installed by no reference script, implemented all the same — through the drop-in classes with the
    kernel wrappers emulated, against goldens produced by the reference's own classes (oracle/make_golden.py)."""
    import emulated_ops
    from oracle import golden

    emulated_ops.install(monkeypatch)
    import adapter.attention_processor as ap
    from imagdressing_b200.modeling import Attention

    gold = golden.load_processors()

    def load(module, prefix):
        module.load_state_dict({k[len(prefix) + 3:]: v.float() for k, v in gold.items() if k.startswith(prefix + ".w.")})
        return module

    rel = lambda a, b: float((a.float() - b.float()).norm() / b.float().norm())
    name = "down_blocks.0.attentions.0.transformer_blocks.0.attn1.processor"
    name2 = name.replace("attn1", "attn2")
    C, H = 160, 4
    attn, attn2 = load(Attention(C, None, H), "refs"), load(Attention(C, 256, H), "cattn")
    x, g2, t = gold["refs.x"], gold["sattn.g"], gold["cattn.t"]
    sp = ap.SAttnProcessor2_0(name, C)
    assert rel(sp(attn, x, sa_hidden_states={name: g2}), gold["sattn.out_g"]) < 1e-2
    assert rel(sp(attn, x), gold["sattn.out_nosa"]) < 1e-2
    rc = load(ap.RefCAttnProcessor2_0(name2, C, 256, scale=0.7), "refc.proc")
    assert rel(rc(attn2, x, encoder_hidden_states=t, sa_hidden_states={name2: g2}), gold["refc.out"]) < 1e-2
    assert rel(rc(attn2, x, encoder_hidden_states=t), gold["refc.out_nosa"]) < 1e-2
    assert set(rc.state_dict()) == {"to_k_ref.weight", "to_v_ref.weight"}
