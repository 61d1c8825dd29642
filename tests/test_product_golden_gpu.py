"""GPU: the drop-in adapter/attention_processor.py + adapter/resampler.py (CUDA kernels through the C ABI) against
the golden vectors produced by the reference's own code. Operands are bf16-exact in the fixture, so the only
difference is arithmetic: tolerance rel-L2 <= 1e-2 (SURVEY.md §8c)."""

import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu
NAME = "down_blocks.0.attentions.0.transformer_blocks.0.attn1.processor"
TOL = 1e-2


@pytest.fixture(scope="module")
def gold(cuda_device):
    from oracle import golden

    return golden.load_processors(cuda_device)


def load(module, gold, prefix, dev):
    sd = {k[len(prefix) + 3:]: v.float() for k, v in gold.items() if k.startswith(prefix + ".w.")}
    module.load_state_dict(sd)
    return module.to(dev)


@torch.no_grad()
def test_processors_vs_reference_goldens(cuda_device, gold):
    import adapter.attention_processor as ap
    from imagdressing_b200.modeling import Attention

    dev = cuda_device
    C, H = 160, 4
    attn = load(Attention(C, None, H), gold, "refs", dev)
    attn2 = load(Attention(C, 256, H), gold, "cattn", dev)
    x, g = gold["refs.x"], gold["refs.g"]  # bf16
    p = load(ap.RefSAttnProcessor2_0(NAME, C, scale=0.9), gold, "refs.proc", dev)
    assert rel_l2(p(attn, x, sa_hidden_states={NAME: g}), gold["refs.out"]) < TOL
    assert rel_l2(p(attn, x), gold["refs.out_nosa"]) < TOL
    cache = ap.CacheAttnProcessor2_0()
    assert rel_l2(cache(attn, x), gold["cache.out"]) < TOL
    assert cache.cache["hidden_states"] is x
    c = ap.CAttnProcessor2_0(NAME, C, 256)
    assert rel_l2(c(attn2, gold["cattn.x"], encoder_hidden_states=gold["cattn.t"], sa_hidden_states={NAME: g}),
                  gold["cattn.out"]) < TOL
    lp = load(ap.LoraRefSAttnProcessor2_0(NAME, C, scale=0.8, rank=16, lora_scale=0.2), gold, "lorarefs.proc", dev)
    assert rel_l2(lp(attn, x, sa_hidden_states={NAME: g}), gold["lorarefs.out"]) < TOL
    rl = load(ap.RefLoraSAttnProcessor2_0(NAME, C, scale=0.8, rank=16, lora_scale=0.2), gold, "lorarefs.proc", dev)
    assert rel_l2(rl(attn, x, sa_hidden_states={NAME: g}), gold["reflora.out"]) < TOL
    ip = load(ap.LoRAIPAttnProcessor2_0(C, 256, rank=16, lora_scale=0.2, scale=0.9, num_tokens=4), gold, "loraip.proc", dev)
    assert rel_l2(ip(attn2, x, encoder_hidden_states=gold["loraip.t"]), gold["loraip.out"]) < TOL
    assert rel_l2(ip(attn2, x, encoder_hidden_states=gold["cattn.t"]), gold["loraip.out_noface"]) < TOL  # quirk B11
    # the two classes no reference script installs: concat-KV single softmax, cross-attention + reference branch
    sp = ap.SAttnProcessor2_0(NAME, C).to(dev)
    assert rel_l2(sp(attn, x, sa_hidden_states={NAME: gold["sattn.g"]}), gold["sattn.out_g"]) < TOL
    assert rel_l2(sp(attn, x), gold["sattn.out_nosa"]) < TOL
    name2 = NAME.replace("attn1", "attn2")
    rc = load(ap.RefCAttnProcessor2_0(name2, C, 256, scale=0.7), gold, "refc.proc", dev)
    assert rel_l2(rc(attn2, x, encoder_hidden_states=gold["cattn.t"], sa_hidden_states={name2: gold["sattn.g"]}),
                  gold["refc.out"]) < TOL
    assert rel_l2(rc(attn2, x, encoder_hidden_states=gold["cattn.t"]), gold["refc.out_nosa"]) < TOL
    # mutable scales take effect (set_scale / set_ipa_scale path): scale 0 == no second stream
    p.scale = 0.0
    assert rel_l2(p(attn, x, sa_hidden_states={NAME: g}), gold["refs.out_nosa"]) < TOL
    # fp16 callers (the reference scripts run fp16) get fp16 back
    assert p(attn, x.half()).dtype == torch.float16


@torch.no_grad()
def test_resampler_vs_reference_goldens(cuda_device, gold):
    from adapter.resampler import ProjPlusModel, Resampler

    dev = cuda_device
    rs = load(Resampler(dim=128, depth=2, dim_head=64, heads=2, num_queries=16, embedding_dim=256, output_dim=128),
              gold, "resampler", dev)
    assert rel_l2(rs(gold["resampler.x"]), gold["resampler.out"]) < TOL
    pp = load(ProjPlusModel(128, 64, 256, 4), gold, "projplus", dev)
    assert rel_l2(pp(gold["projplus.id"], gold["projplus.clip"]), gold["projplus.out"]) < TOL
    assert rel_l2(pp(gold["projplus.id"], gold["projplus.clip"], shortcut=True, scale=0.5),
                  gold["projplus.out_shortcut"]) < TOL
