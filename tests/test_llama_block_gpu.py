"""GPU: the LLaMA frozen-block fast path (lm_blocks.FastLlamaBlock) and its kernels -- RMSNorm, RoPE, the SwiGLU GEMM
epilogue and its backward -- against torch and HF's own LlamaDecoderLayer (the LM is third-party code; HF's module IS
the reference for it).  Block tolerances as for MPT (test_lm_block_gpu.py): outputs 2e-2 of max, input gradients
4e-2 of max, cosine >= 0.999."""
import pytest
import torch

from test_lm_block_gpu import cmp

pytestmark = pytest.mark.gpu

bf16 = torch.bfloat16
VIT = dict(image_size=56, patch_size=14, width=128, layers=2, heads=2, output_dim=128)


def llama_cfg(D, heads, I, kv=None, **kw):
    from transformers import LlamaConfig
    cfg = LlamaConfig(hidden_size=D, num_attention_heads=heads, num_key_value_heads=kv or heads, intermediate_size=I,
                      num_hidden_layers=1, vocab_size=61, max_position_embeddings=512, **kw)
    cfg._attn_implementation = "sdpa"
    return cfg


def make_block(D, heads, I, seed, **kw):
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer, LlamaRotaryEmbedding
    torch.manual_seed(seed)
    cfg = llama_cfg(D, heads, I, **kw)
    blk = LlamaDecoderLayer(cfg, 0).cuda().eval().requires_grad_(False)
    with torch.no_grad():
        for _, p in blk.named_parameters():
            if p.dim() == 1:
                p.copy_(1.0 + 0.1 * torch.randn_like(p))
            else:
                p.copy_(torch.randn_like(p) * p.shape[1] ** -0.5)
    return blk, LlamaRotaryEmbedding(cfg).cuda()


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("D", [256, 4096])
def test_rmsnorm_fwd_bwd(D):
    from open_flamingo_b200 import ops
    rows = 333
    torch.manual_seed(0)
    x = torch.randn(rows, D, device="cuda") * 3
    w = 1 + 0.1 * torch.randn(D, device="cuda")
    dx_add = torch.randn(rows, D, device="cuda")
    xr = x.clone().requires_grad_(True)
    ref = w * (xr * torch.rsqrt(xr.pow(2).mean(-1, keepdim=True) + 1e-5))
    y, rstd = ops.rmsnorm_fwd(x, w, 1e-5)
    cmp(y, ref.to(bf16), 1e-2, "rmsnorm y")
    assert torch.allclose(rstd, torch.rsqrt(x.pow(2).mean(-1) + 1e-5), rtol=1e-5)
    dy = torch.randn(rows, D, device="cuda").to(bf16)
    ref.backward(dy.float())
    dx = ops.rmsnorm_bwd(dy, x, w, rstd, dx_add=dx_add)
    assert torch.allclose(dx, xr.grad + dx_add, rtol=1e-4, atol=1e-4 * xr.grad.abs().max().item())


def _rope_inputs(B, T, heads, hd, cs_batch, rope_kw, seed):
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding
    torch.manual_seed(seed)
    D = heads * hd
    cfg = llama_cfg(D, heads, 64, **rope_kw)
    rot = LlamaRotaryEmbedding(cfg).cuda()
    pos = torch.arange(T, device="cuda").view(1, T).expand(cs_batch, T) + \
        torch.arange(cs_batch, device="cuda").view(cs_batch, 1) * 7
    cos, sin = rot(torch.zeros(1, device="cuda"), pos)
    qkv = torch.randn(B * T, 3 * D, device="cuda").to(bf16)
    return qkv, cos, sin


def _heads(t, B, T, heads, hd):
    return t.view(B, T, heads, hd).transpose(1, 2)


ROPES = [dict(), dict(rope_parameters=dict(rope_type="llama3", rope_theta=500000.0, factor=8.0, low_freq_factor=1.0,
                                           high_freq_factor=4.0, original_max_position_embeddings=64))]


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("cs_batch", [1, 3])
@pytest.mark.parametrize("rope", [0, 1])
def test_rope_matches_hf(hd, cs_batch, rope):
    from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
    from open_flamingo_b200 import ops
    B, T, heads = 3, 40, 2
    D = heads * hd
    qkv, cos, sin = _rope_inputs(B, T, heads, hd, cs_batch, ROPES[rope], 1)
    q = _heads(qkv[:, :D], B, T, heads, hd)
    k = _heads(qkv[:, D:2 * D], B, T, heads, hd)
    qr, kr = apply_rotary_pos_emb(q, k, cos, sin)
    got = qkv.clone()
    ops.rope_(got, B, T, 2 * heads, hd, cos.contiguous(), sin.contiguous())
    for g, r in ((got[:, :D], qr), (got[:, D:2 * D], kr)):
        g = _heads(g, B, T, heads, hd).float()
        r = r.to(bf16).float()
        ulp = (r.abs().clamp_min(1e-30).log2().floor() - 7).exp2()     # 1 bf16 ulp
        assert ((g - r).abs() <= ulp).all(), (g - r).abs().max()
    assert torch.equal(got[:, 2 * D:], qkv[:, 2 * D:])                  # v untouched

    # inverse = autograd of HF's rope on the same bf16 inputs
    qg = q.detach().clone().requires_grad_(True)
    kg = k.detach().clone().requires_grad_(True)
    qr, kr = apply_rotary_pos_emb(qg, kg, cos, sin)
    dq = torch.randn_like(qr).to(bf16)
    dk = torch.randn_like(kr).to(bf16)
    (qr * dq.float()).sum().backward()
    (kr * dk.float()).sum().backward()
    d = torch.zeros_like(qkv)
    d[:, :D] = dq.transpose(1, 2).reshape(B * T, D)
    d[:, D:2 * D] = dk.transpose(1, 2).reshape(B * T, D)
    ops.rope_(d, B, T, 2 * heads, hd, cos.contiguous(), sin.contiguous(), inverse=True)
    cmp(_heads(d[:, :D], B, T, heads, hd), qg.grad, 1e-2, "rope inverse q")
    cmp(_heads(d[:, D:2 * D], B, T, heads, hd), kg.grad, 1e-2, "rope inverse k")


@pytest.mark.parametrize("M", [200, 1100])          # cta_group::1 and ::2 kernels
@pytest.mark.parametrize("I", [352, 1024])          # 352: not a multiple of 256
def test_swiglu_gemm_and_bwd(M, I):
    from open_flamingo_b200 import lm_blocks, ops
    K = 256
    torch.manual_seed(2)
    x = torch.randn(M, K, device="cuda").to(bf16)
    wg = (torch.randn(I, K, device="cuda") * K ** -0.5).to(bf16)
    wu = (torch.randn(I, K, device="cuda") * K ** -0.5).to(bf16)
    wp = lm_blocks.pack_gate_up(wg, wu).contiguous()
    h, gu = ops.swiglu_gemm(x, wp)
    g = (x.float() @ wg.float().t()).to(bf16)
    u = (x.float() @ wu.float().t()).to(bf16)
    ref = (torch.nn.functional.silu(g) * u)
    cmp(h, ref, 1e-2, "swiglu h")
    g2, u2 = lm_blocks.unpack_gate_up(gu.t())
    cmp(g2.t(), g, 1e-2, "swiglu raw g")
    cmp(u2.t(), u, 1e-2, "swiglu raw u")
    # backward against autograd on the same bf16 g / u
    gg = g2.t().contiguous().requires_grad_(True)
    uu = u2.t().contiguous().requires_grad_(True)
    hh = torch.nn.functional.silu(gg) * uu
    dh = torch.randn_like(hh)
    hh.backward(dh)
    dgu = ops.swiglu_bwd(dh, gu)
    dg, du = lm_blocks.unpack_gate_up(dgu.t())
    cmp(dg.t(), gg.grad, 1e-2, "swiglu dg")
    cmp(du.t(), uu.grad, 1e-2, "swiglu du")
    # one packed dgrad GEMM = gate dgrad + up dgrad
    dx = ops.gemm(dgu, wp, b_mn=True)
    cmp(dx, gg.grad.float() @ wg.float() + uu.grad.float() @ wu.float(), 2e-2, "packed dgrad")


# ------------------------------------------------------------------------------------------------ block parity
def hf_mask(B, T, kind, dtype_ref):
    from transformers.masking_utils import create_causal_mask
    att = torch.ones(B, T, dtype=torch.long, device="cuda")
    if kind == "right_pad":
        att[0, T - 7:] = 0
    elif kind == "left_pad":
        att[1, :5] = 0
    cfg = llama_cfg(64, 1, 64)
    emb = torch.zeros(B, T, 64, device="cuda", dtype=dtype_ref)
    pos = torch.arange(T, device="cuda").view(1, T)
    m = create_causal_mask(config=cfg, inputs_embeds=emb, attention_mask=None if kind == "causal" else att,
                           past_key_values=None, position_ids=pos)
    return m, att


def run_hf(blk, x, mask, pe, autocast):
    # SDPA's defined result for a query with no allowed key is a zero output (math and memory-efficient backends,
    # and the CPU).  torch's cuDNN backend, which it prefers for bf16 with a mask on the B200, returns nonzero values
    # for such rows instead, so the reference is computed on the backends that implement the definition.
    from torch.nn.attention import SDPBackend, sdpa_kernel
    with sdpa_kernel([SDPBackend.EFFICIENT_ATTENTION, SDPBackend.MATH]), \
            torch.autocast("cuda", dtype=bf16, enabled=autocast):
        return blk(x, attention_mask=mask, position_embeddings=pe)


@pytest.mark.parametrize("D,heads", [(256, 4), (256, 2)])    # head_dim 64 and 128
@pytest.mark.parametrize("kind", ["causal", "right_pad", "left_pad"])
@pytest.mark.parametrize("T", [96, 130])
def test_fast_llama_block_matches_hf(D, heads, kind, T):
    from open_flamingo_b200 import lm_blocks
    blk, rot = make_block(D, heads, 688, 3)
    fast = lm_blocks.accelerate(blk)
    assert isinstance(fast, lm_blocks.FastLlamaBlock)
    B = 2
    torch.manual_seed(4)
    x = torch.randn(B, T, D, device="cuda")
    mask, att = hf_mask(B, T, kind, torch.float32)
    pos = torch.arange(T, device="cuda").view(1, T)
    pe = rot(x, pos)
    flag = att.all().to(torch.int32).reshape(1)
    w = torch.randn(B, T, D, device="cuda")
    outs, grads = {}, {}
    for name in ("autocast", "fp32", "fast"):
        xg = x.clone().requires_grad_(True)
        if name == "fast":
            with torch.autocast("cuda", dtype=bf16):
                y = fast(xg, attention_mask=mask, position_embeddings=pe, pure_causal_flag=flag)
            assert y is not None, "fast path declined"
        else:
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            try:
                y = run_hf(blk, xg, mask, pe, name == "autocast")
            finally:
                torch.backends.cuda.matmul.allow_tf32 = prev
        (y * w).sum().backward()
        outs[name], grads[name] = y.detach().float(), xg.grad.float()
    cmp(outs["fast"], outs["autocast"], 2e-2, f"block out [{kind}]")
    cmp(grads["fast"], grads["autocast"], 4e-2, f"block dx [{kind}]")
    # DESIGN.md section 2: no further from fp32 than the autocast reference is
    for what, d in (("out", outs), ("dx", grads)):
        e_ours = (d["fast"] - d["fp32"]).abs().max().item()
        e_ac = (d["autocast"] - d["fp32"]).abs().max().item()
        assert e_ours <= 2 * e_ac + 1e-6, f"{what} [{kind}]: ours {e_ours:.3e} vs autocast {e_ac:.3e}"
    if kind == "left_pad":
        # query rows with no allowed key: SDPA gives a zero attention output, so the block adds only the MLP branch
        dead = ~mask[1, 0].any(-1)
        assert dead.sum().item() == 5
        assert torch.allclose(outs["fast"][1, dead], outs["autocast"][1, dead], rtol=2e-2, atol=2e-2)


def test_fast_llama_declines():
    from open_flamingo_b200 import lm_blocks
    blk, rot = make_block(256, 4, 688, 5)
    fast = lm_blocks.accelerate(blk)
    x = torch.randn(1, 8, 256, device="cuda")
    pe = rot(x, torch.arange(8, device="cuda").view(1, 8))
    assert fast(x, position_embeddings=pe) is not None
    assert fast(x, position_embeddings=pe, output_attentions=True) is None
    assert fast(x, position_embeddings=pe, use_cache=True) is None
    assert fast(x, position_embeddings=pe, attention_mask=torch.zeros(1, 1, 8, 8, device="cuda")) is None
    blk.mlp.up_proj.weight.requires_grad_(True)
    assert fast(x, position_embeddings=pe) is None
    gqa, rot2 = make_block(256, 4, 688, 6, kv=2)
    pe2 = rot2(x, torch.arange(8, device="cuda").view(1, 8))
    assert lm_blocks.accelerate(gqa)(x, position_embeddings=pe2) is None


def test_weight_cache_follows_load_state_dict():
    from open_flamingo_b200 import lm_blocks
    blk, rot = make_block(256, 4, 688, 7)
    fast = lm_blocks.accelerate(blk)
    x = torch.randn(2, 16, 256, device="cuda")
    pe = rot(x, torch.arange(16, device="cuda").view(1, 16))
    with torch.autocast("cuda", dtype=bf16):
        y0 = fast(x, position_embeddings=pe)
    other, _ = make_block(256, 4, 688, 8)
    blk.load_state_dict(other.state_dict())
    with torch.autocast("cuda", dtype=bf16):
        y1 = fast(x, position_embeddings=pe)
        ref = blk(x, position_embeddings=pe)
    assert not torch.allclose(y0, y1)
    cmp(y1, ref, 2e-2, "after load_state_dict")


# ------------------------------------------------------------------------------------------------ full model
LLAMA = dict(hidden_size=128, num_hidden_layers=4, num_attention_heads=2, num_key_value_heads=2, intermediate_size=352,
             vocab_size=61, max_position_embeddings=128)


def build(seed=0, **over):
    from open_flamingo_b200.testing import build_flamingo, build_llama, synthetic_batch
    model, _, tok = build_flamingo(VIT, dict(LLAMA, **over), cross_attn_every_n_layers=2, device="cuda", gate_init=1.0,
                                   seed=seed, lm_builder=build_llama)
    media_id, eoc_id = tok.encode("<image>")[-1], tok.encode("<|endofchunk|>")[-1]
    batch = {k: v.cuda() for k, v in synthetic_batch(3, 2, 24, media_id, eoc_id, 61, image_size=56, seed=9).items()}
    return model, batch


def fwd_bwd(model, batch):
    with torch.autocast("cuda", dtype=bf16):
        out = model(vision_x=batch["vision_x"], lang_x=batch["lang_x"], attention_mask=batch["attention_mask"],
                    labels=batch["labels"])
    out.loss.backward()
    return out


def test_full_model_fast_path_on_and_off(monkeypatch):
    from transformers.models.llama import modeling_llama
    from open_flamingo_b200 import lm_blocks
    model, batch = build(seed=1)
    model.train()
    batch["attention_mask"][0, -5:] = 0           # one right-padded row
    res = {}
    for on in (True, False):
        model.zero_grad(set_to_none=True)
        lm_blocks.ENABLED = on
        try:
            with monkeypatch.context() as mp:
                if on:   # the fast path must really run: HF's block forward may not be called
                    def boom(*a, **k):
                        raise AssertionError("LlamaDecoderLayer.forward ran with the fast path enabled")
                    mp.setattr(modeling_llama.LlamaDecoderLayer, "forward", boom)
                out = fwd_bwd(model, batch)
        finally:
            lm_blocks.ENABLED = True
        grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.requires_grad}
        res[on] = (out.logits.detach(), out.loss.detach(), grads)
    cmp(res[True][0], res[False][0], 2e-2, "logits")
    assert abs(res[True][1].item() - res[False][1].item()) <= 2e-2 * abs(res[False][1].item())
    for n in res[False][2]:
        cmp(res[True][2][n], res[False][2][n], 4e-2, f"grad {n}")

    model.eval()
    prompt = batch["lang_x"][:1, :8]
    vis = batch["vision_x"][:1]
    toks = {}
    for on in (True, False):
        lm_blocks.ENABLED = on
        try:
            with torch.no_grad(), torch.autocast("cuda", dtype=bf16):
                toks[on] = model.generate(vis, prompt, attention_mask=torch.ones_like(prompt), max_new_tokens=6,
                                          num_beams=1, do_sample=False)
        finally:
            lm_blocks.ENABLED = True
    assert torch.equal(toks[True], toks[False])


def test_gqa_flamingo_runs_through_hf_blocks():
    from open_flamingo_b200 import lm_blocks
    model, batch = build(seed=2, num_key_value_heads=1)
    blk = model.lang_encoder._get_decoder_layers()[0]
    assert blk._fast_block is not None
    out = fwd_bwd(model.train(), batch)
    assert torch.isfinite(out.loss)
    assert lm_blocks.llama_decline_reason(blk.decoder_layer, torch.zeros(1, 4, 128, device="cuda")) == \
        "grouped-query attention"


def test_graphed_step_equals_eager_step():
    import copy
    from open_flamingo_b200.train import FlatTrainer, GraphedTrainStep
    m1, batch = build(seed=1)
    m1.train()
    m2 = copy.deepcopy(m1)
    t1 = FlatTrainer(m1, lr=1e-3)
    losses_eager = []
    for _ in range(4):
        t1.zero_grad()
        losses_eager.append(fwd_bwd(m1, batch).loss.detach().item())
        t1.step()
    t1.close()
    t2 = FlatTrainer(m2, lr=1e-3)
    g = GraphedTrainStep(m2, t2, batch, warmup=1)
    assert g.ok, getattr(g, "traceback", g.error)
    losses_graph = [losses_eager[0]] + [g(batch).item() for _ in range(3)]
    for a, b in zip(losses_eager[1:], losses_graph[1:]):
        assert abs(a - b) <= 2e-2 * abs(a) + 1e-3, (losses_eager, losses_graph)
