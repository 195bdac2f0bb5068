"""CPU: host side of the LLaMA frozen-block fast path -- factory wiring, dispatch, the decline rules, the gate/up
packing helper, and a static SASS check of the SwiGLU GEMM instances in the shipped library."""
import re

import pytest
import torch

from test_abi_cpu import _sass_by_kernel

VIT = dict(image_size=56, patch_size=14, width=128, layers=2, heads=2, output_dim=128)
LLAMA = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=2, intermediate_size=352,
             vocab_size=61, max_position_embeddings=128)


def make_block(**over):
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer
    kw = dict(LLAMA, **over)
    cfg = LlamaConfig(**kw)
    cfg._attn_implementation = "sdpa"
    return LlamaDecoderLayer(cfg, 0).eval().requires_grad_(False)


def reason(blk, T=8, cos_dim=None, mask=None, **kw):
    from open_flamingo_b200 import lm_blocks
    D = blk.hidden_size
    hd = blk.self_attn.head_dim
    x = torch.randn(2, T, D)
    cs = torch.randn(1, T, cos_dim or hd)
    return lm_blocks.llama_decline_reason(blk, x, mask, (cs, cs.clone()), **kw)


def test_factory_wraps_every_llama_block():
    from open_flamingo_b200 import lm_blocks
    from open_flamingo_b200.testing import build_flamingo, build_llama
    model, _, _ = build_flamingo(VIT, LLAMA, cross_attn_every_n_layers=2, device="cpu", lm_builder=build_llama)
    lm = model.lang_encoder
    assert lm.decoder_layers_attr_name == "model.layers"
    layers = lm._get_decoder_layers()
    assert len(layers) == 2
    assert all(isinstance(layer._fast_block, lm_blocks.FastLlamaBlock) for layer in layers)
    assert [layer.gated_cross_attn_layer is not None for layer in layers] == [False, True]


def test_accelerate_dispatch():
    from open_flamingo_b200 import lm_blocks
    blk = make_block()
    assert isinstance(lm_blocks.accelerate(blk), lm_blocks.FastLlamaBlock)
    assert lm_blocks.accelerate(torch.nn.Linear(4, 4)) is None
    assert lm_blocks.accelerate(blk.mlp) is None


def test_supported_block_declines_only_for_the_device():
    assert reason(make_block()) == "not on CUDA"
    assert reason(make_block(num_attention_heads=1, num_key_value_heads=1)) == "not on CUDA"   # head_dim 128
    assert reason(make_block(), mask=torch.ones(2, 1, 8, 8, dtype=torch.bool)) == "not on CUDA"
    assert reason(make_block(), mask=torch.ones(1, 1, 8, 8, dtype=torch.bool)) == "not on CUDA"


@pytest.mark.parametrize("case,expect", [
    ("gqa", "grouped-query"),
    ("attention_bias", "bias"),
    ("mlp_bias", "bias"),
    ("gelu", "hidden_act"),
    ("head_dim_32", "head_dim"),
    ("partial_rotary", "partial rotary"),
    ("trainable", "trainable"),
    ("past_key_values", "KV cache"),
    ("use_cache", "KV cache"),
    ("output_attentions", "output_attentions"),
    ("float_mask", "float"),
    ("dropout", "dropout"),
    ("scaling", "scaling"),
    ("wide", "hidden size"),
])
def test_decline_rules(case, expect):
    kw, blk = {}, None
    if case == "gqa":
        blk = make_block(num_attention_heads=2, num_key_value_heads=1)
    elif case == "attention_bias":
        blk = make_block(attention_bias=True)
    elif case == "mlp_bias":
        blk = make_block(mlp_bias=True)
    elif case == "gelu":
        blk = make_block(hidden_act="gelu")
    elif case == "head_dim_32":
        blk = make_block(num_attention_heads=4, num_key_value_heads=4)
    elif case == "partial_rotary":
        kw["cos_dim"] = 32
    elif case == "trainable":
        blk = make_block()
        blk.mlp.up_proj.weight.requires_grad_(True)
    elif case == "past_key_values":
        kw["past_key_values"] = object()
    elif case == "use_cache":
        kw["use_cache"] = True
    elif case == "output_attentions":
        kw["output_attentions"] = True
    elif case == "float_mask":
        kw["mask"] = torch.zeros(2, 1, 8, 8)
    elif case == "dropout":
        blk = make_block(attention_dropout=0.1).train()
    elif case == "scaling":
        blk = make_block()
        blk.self_attn.scaling = 0.5
    elif case == "wide":
        blk = make_block(hidden_size=8192, num_attention_heads=64, num_key_value_heads=64, intermediate_size=32)
    r = reason(blk if blk is not None else make_block(), **kw)
    assert r is not None and expect in r, r


def test_gate_up_packing_layout_and_round_trip():
    from open_flamingo_b200 import lm_blocks
    I, D = 48, 5
    g = torch.arange(I * D, dtype=torch.float32).view(I, D)
    u = -torch.arange(I * D, dtype=torch.float32).view(I, D) - 1
    p = lm_blocks.pack_gate_up(g, u)
    assert p.shape == (2 * I, D)
    for j in range(I // 16):
        assert torch.equal(p[32 * j:32 * j + 16], g[16 * j:16 * j + 16])
        assert torch.equal(p[32 * j + 16:32 * j + 32], u[16 * j:16 * j + 16])
    g2, u2 = lm_blocks.unpack_gate_up(p)
    assert torch.equal(g2, g) and torch.equal(u2, u)
    # the packed activations [R, 2I] unpack through their transpose
    gu = p.t().contiguous()
    g3, u3 = lm_blocks.unpack_gate_up(gu.t())
    assert torch.equal(g3, g) and torch.equal(u3, u)
    with pytest.raises(ValueError):
        lm_blocks.pack_gate_up(g[:40], u[:40])


def test_swiglu_gemm_instances_are_tcgen05_and_tma():
    import __graft_entry__ as g
    g.build()
    kernels = _sass_by_kernel()
    # EPI id 10 = OFK_EPI_SWIGLU_DUAL: the 1-CTA kernel at both tile widths and the 2-CTA kernel, K-major operands
    swiglu = {k: v for k, v in kernels.items()
              if re.search(r"gemm_kernelILi(128|256)ELi0ELi0ELi10EE|gemm2_kernelILi0ELi0ELi10EE", k)}
    assert len(swiglu) == 3, sorted(swiglu)
    for k, ops_ in swiglu.items():
        assert "UTCHMMA" in ops_, f"{k}: no tcgen05.mma"
        assert "LDTM" in ops_, f"{k}: accumulators are not read from TMEM"
        assert "UTMALDG" in ops_, f"{k}: operands are not staged by TMA"
        assert "HMMA" not in ops_, f"{k}: mma.sync inside a tcgen05 kernel"
    assert any("rope_kernel" in k for k in kernels) and any("swiglu_bwd_kernel" in k for k in kernels)
