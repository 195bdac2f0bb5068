"""Frozen-LM decoder blocks on the sm_100a kernels (SURVEY.md section 8f, rank 1).

The reference runs the frozen LM's decoder block as ordinary PyTorch (`self.decoder_layer(lang_x, ...)`,
flamingo_lm.py:63-65).  Two LM families are evaluated with the kernels already used by the gated blocks (tcgen05
GEMMs with fused epilogues, LayerNorm / RMSNorm, dense attention), forward plus the dgrad-only backward a frozen
block needs:
  MPT   (HF `MptBlock`, named by BASELINE.json): LN -> Wqkv -> causal ALiBi attention -> out_proj -> +res -> LN ->
        up_proj -> GELU(erf) -> down_proj -> +res, no biases;
  LLaMA (HF `LlamaDecoderLayer`, OpenFlamingo-9B v1): RMSNorm -> q/k/v_proj -> RoPE -> causal attention -> o_proj ->
        +res -> RMSNorm -> silu(gate_proj) * up_proj -> down_proj -> +res, no biases.
Anything else -- other LM families, KV-cache decoding, dropout, GQA, output_attentions, ... -- takes the block's own
PyTorch forward, exactly as in the reference.

Numerics are those of the block under `torch.autocast(bfloat16)`: fp32 residual stream, fp32 norm statistics and
softmax, bf16 GEMM operands.
"""
import weakref

import torch

from . import _lib as L
from . import ops
from .fused import w16

bf16 = torch.bfloat16
f32 = torch.float32

ENABLED = True  # module-level switch (bench.py --lm eager turns it off to time the reference's PyTorch LM path)

_zero_bias = {}
_mask_cache = [None, None]  # (weakref to HF's [B,1,T,T] bool mask, its contiguous [B,T,T] byte view) -- one per forward


def _zeros(n, device):
    key = (n, device)
    t = _zero_bias.get(key)
    if t is None:
        t = torch.zeros(n, device=device, dtype=f32)
        _zero_bias[key] = t
    return t


class FrozenMptBlockFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mask, pure_flag, slopes, heads, eps, n1_w, wqkv, wout, n2_w, wup, wdown):
        B, T, D = x.shape
        R = B * T
        hd = D // heads
        x2d = x.reshape(R, D)
        if not x2d.is_contiguous():
            x2d = x2d.contiguous()
        zb = _zeros(D, x.device)
        xn, mean1, rstd1 = ops.layernorm_fwd(x2d, n1_w, zb, eps)
        qkv = ops.gemm(xn, w16(wqkv))                                               # [R, 3D]
        del xn
        q3 = qkv.view(B, T, 3 * D)
        scale = float(hd ** -0.5)
        o, lse = ops.attn_dense_fwd(q3[..., :D], q3[..., D:2 * D], q3[..., 2 * D:], heads, hd, scale,
                                    causal=mask is None, mask=mask, slopes=slopes, pure_causal_flag=pure_flag)
        x1 = ops.gemm(o.view(R, D), w16(wout), epi=L.EPI_GATE_RESID_F32, aux=x2d)   # + residual
        x1n, mean2, rstd2 = ops.layernorm_fwd(x1, n2_w, zb, eps)
        z = torch.empty((R, wup.shape[0]), device=x.device, dtype=bf16)
        h = torch.empty((R, wup.shape[0]), device=x.device, dtype=bf16)
        ops.gemm(x1n, w16(wup), epi=L.EPI_GELU_DUAL, out=z, out2=h)
        del x1n
        out = ops.gemm(h, w16(wdown), epi=L.EPI_GATE_RESID_F32, aux=x1)             # + residual
        del h
        ctx.save_for_backward(x2d, mean1, rstd1, qkv, o, lse, x1, mean2, rstd2, z, n1_w, wqkv, wout, n2_w, wup,
                              wdown, slopes, mask if mask is not None else x2d.new_empty(0),
                              pure_flag if pure_flag is not None else x2d.new_empty(0))
        ctx.meta = (B, T, D, heads, hd, scale, mask is not None, pure_flag is not None)
        return out.view(B, T, D)

    @staticmethod
    def backward(ctx, dout):
        (x2d, mean1, rstd1, qkv, o, lse, x1, mean2, rstd2, z, n1_w, wqkv, wout, n2_w, wup, wdown, slopes,
         mask, pure_flag) = ctx.saved_tensors
        B, T, D, heads, hd, scale, has_mask, has_flag = ctx.meta
        if not has_mask:
            mask = None
        if not has_flag:
            pure_flag = None
        R = B * T
        d2 = dout.reshape(R, D)
        if not d2.is_contiguous():
            d2 = d2.contiguous()
        if d2.dtype != f32:
            d2 = d2.float()
        dbr = ops.gate_bwd(d2, None, None, None)                                    # bf16 cast
        dz = ops.gemm(dbr, w16(wdown), b_mn=True, epi=L.EPI_DGELU_BF16, aux=z)      # (d W_down) * gelu'(z)
        dx1n = ops.gemm(dz, w16(wup), b_mn=True)
        del dz, dbr
        dx1 = ops.layernorm_bwd(dx1n, x1, n2_w, mean2, rstd2, dx_add=d2)
        da = ops.gate_bwd(dx1, None, None, None)
        d_o = ops.gemm(da, w16(wout), b_mn=True)                                    # [R, D]
        del da
        q3 = qkv.view(B, T, 3 * D)
        dqkv = torch.empty_like(qkv)
        dq3 = dqkv.view(B, T, 3 * D)
        ops.attn_dense_bwd(q3[..., :D], q3[..., D:2 * D], q3[..., 2 * D:], o, d_o.view(B, T, D), lse, heads, hd, scale,
                           causal=mask is None, mask=mask, slopes=slopes, pure_causal_flag=pure_flag,
                           dq=dq3[..., :D], dk=dq3[..., D:2 * D], dv=dq3[..., 2 * D:])
        dxn = ops.gemm(dqkv, w16(wqkv), b_mn=True)
        dx = ops.layernorm_bwd(dxn, x2d, n1_w, mean1, rstd1, dx_add=dx1)
        return (dx.view(B, T, D),) + (None,) * 11


def _alibi_slopes(position_bias):
    """HF builds bias[h, 0, k] = slope_h * (k - (L-1)) (build_mpt_alibi_tensor); recover slope_h."""
    pb = position_bias
    if pb.dim() != 3 or pb.shape[-1] < 2:
        return None
    return (pb[:, 0, -1] - pb[:, 0, -2]).float().contiguous()


class FastMptBlock:
    """Callable with HF MptBlock.forward's signature; returns None when the fast path does not apply."""

    def __init__(self, block):
        self.block = block
        self._slopes = None

    def applicable(self, hidden_states, position_bias, attention_mask, layer_past, use_cache, output_attentions):
        b = self.block
        if not ENABLED or not hidden_states.is_cuda or layer_past is not None or output_attentions:
            return False
        if use_cache:
            return False   # a caller that wants a `present` back (tuple-cache HF versions) gets the block's own forward
        a = b.attn
        if getattr(a, "clip_qkv", None) or (b.training and (a.attn_dropout_p > 0 or b.dropout_rate > 0 or
                                                            b.ffn.hidden_dropout > 0)):
            return False
        if a.head_dim not in (64, 128) or position_bias is None:
            return False
        if a.Wqkv.bias is not None or a.out_proj.bias is not None or b.ffn.up_proj.bias is not None or \
                b.ffn.down_proj.bias is not None or b.norm_1.bias is not None or b.norm_2.bias is not None:
            return False
        if any(p.requires_grad for p in b.parameters()):
            return False  # this path has no wgrad: frozen blocks only
        if not isinstance(b.ffn.act, torch.nn.GELU) or b.ffn.act.approximate != "none":
            return False
        if abs(a.softmax_scale - a.head_dim ** -0.5) > 1e-9:
            return False
        return True

    def __call__(self, hidden_states, position_bias=None, attention_mask=None, layer_past=None, use_cache=False,
                 output_attentions=False, pure_causal_flag=None, **kwargs):
        if not self.applicable(hidden_states, position_bias, attention_mask, layer_past, use_cache, output_attentions):
            return None
        b = self.block
        a = b.attn
        B, T, D = hidden_states.shape
        if self._slopes is None or self._slopes.device != hidden_states.device:
            self._slopes = _alibi_slopes(position_bias)
            if self._slopes is None:
                return None
        mask = None
        if attention_mask is not None:
            m = attention_mask
            if m.dtype != torch.bool or m.dim() != 4 or m.shape[1] != 1 or m.shape[2] != T or m.shape[3] != T:
                return None
            ref = _mask_cache[0]
            if ref is not None and ref() is m and _mask_cache[1].shape[0] == B:
                mask = _mask_cache[1]
            else:
                mask = m.expand(B, 1, T, T).reshape(B, T, T).contiguous()
                _mask_cache[0], _mask_cache[1] = weakref.ref(m), mask
        x = hidden_states if hidden_states.dtype == f32 else hidden_states.float()
        out = FrozenMptBlockFn.apply(x, mask, pure_causal_flag if mask is not None else None, self._slopes, a.n_heads, b.norm_1.eps, b.norm_1.weight, a.Wqkv.weight,
                                     a.out_proj.weight, b.norm_2.weight, b.ffn.up_proj.weight, b.ffn.down_proj.weight)
        if out.dtype != hidden_states.dtype:
            out = out.to(hidden_states.dtype)
        return out, None


# ---------------------------------------------------------------------------------------------------------------
# LLaMA

_llama_mask_cache = [None, None, None]  # (weakref to HF's [B,1,T,T] bool mask, kernel byte mask [B,T,T], row keep [B,T,1])


def pack_gate_up(w_gate, w_up):
    """[gate_proj; up_proj] rows ([I, ...] each, I % 16 == 0) interleaved in the OFK_SWIGLU_GROUP layout of
    include/ofk.h: packed rows 32j..32j+15 are gate rows 16j..16j+15, packed rows 32j+16..32j+31 the same up rows."""
    G = L.SWIGLU_GROUP
    I = w_gate.shape[0]
    if w_up.shape != w_gate.shape or I % G != 0:
        raise ValueError(f"gate / up must have the same shape with rows % {G} == 0")
    rest = tuple(w_gate.shape[1:])
    return torch.stack((w_gate.reshape(I // G, G, *rest), w_up.reshape(I // G, G, *rest)), 1).reshape(2 * I, *rest)


def unpack_gate_up(packed):
    """Inverse of pack_gate_up along dim 0: returns (gate, up)."""
    G = L.SWIGLU_GROUP
    rest = tuple(packed.shape[1:])
    v = packed.reshape(packed.shape[0] // (2 * G), 2, G, *rest)
    return v[:, 0].reshape(-1, *rest), v[:, 1].reshape(-1, *rest)


class FrozenLlamaBlockFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mask, keep, pure_flag, cos, sin, heads, eps1, eps2, n1_w, wqkv, wo, n2_w, wgu, wdown):
        B, T, D = x.shape
        R = B * T
        hd = D // heads
        x2d = x.reshape(R, D)
        if not x2d.is_contiguous():
            x2d = x2d.contiguous()
        xn, rstd1 = ops.rmsnorm_fwd(x2d, n1_w, eps1)
        qkv = ops.gemm(xn, wqkv)                                                    # [R, 3D]
        del xn
        ops.rope_(qkv, B, T, 2 * heads, hd, cos, sin)                               # q and k in place
        q3 = qkv.view(B, T, 3 * D)
        scale = float(hd ** -0.5)
        o, lse = ops.attn_dense_fwd(q3[..., :D], q3[..., D:2 * D], q3[..., 2 * D:], heads, hd, scale,
                                    causal=mask is None, mask=mask, slopes=None, pure_causal_flag=pure_flag)
        if keep is not None:
            o.mul_(keep)     # a query with no allowed key gets a zero output, as torch SDPA gives it
        x1 = ops.gemm(o.view(R, D), w16(wo), epi=L.EPI_GATE_RESID_F32, aux=x2d)    # + residual
        x1n, rstd2 = ops.rmsnorm_fwd(x1, n2_w, eps2)
        h, gu = ops.swiglu_gemm(x1n, wgu)
        del x1n
        out = ops.gemm(h, w16(wdown), epi=L.EPI_GATE_RESID_F32, aux=x1)             # + residual
        del h
        empty = x2d.new_empty(0)
        ctx.save_for_backward(x2d, rstd1, qkv, o, lse, x1, rstd2, gu, cos, sin, n1_w, wqkv, wo, n2_w, wgu, wdown,
                              empty if mask is None else mask, empty if keep is None else keep,
                              empty if pure_flag is None else pure_flag)
        ctx.meta = (B, T, D, heads, hd, scale, mask is not None, keep is not None, pure_flag is not None)
        return out.view(B, T, D)

    @staticmethod
    def backward(ctx, dout):
        (x2d, rstd1, qkv, o, lse, x1, rstd2, gu, cos, sin, n1_w, wqkv, wo, n2_w, wgu, wdown, mask, keep,
         pure_flag) = ctx.saved_tensors
        B, T, D, heads, hd, scale, has_mask, has_keep, has_flag = ctx.meta
        mask = mask if has_mask else None
        keep = keep if has_keep else None
        pure_flag = pure_flag if has_flag else None
        R = B * T
        d2 = dout.reshape(R, D)
        if not d2.is_contiguous():
            d2 = d2.contiguous()
        if d2.dtype != f32:
            d2 = d2.float()
        dbr = ops.gate_bwd(d2, None, None, None)                                    # bf16 cast
        dh = ops.gemm(dbr, w16(wdown), b_mn=True)                                   # [R, I]
        del dbr
        dgu = ops.swiglu_bwd(dh, gu)                                                # [R, 2I] packed
        del dh
        dx1n = ops.gemm(dgu, wgu, b_mn=True)                                        # gate and up dgrad in one GEMM
        del dgu
        dx1 = ops.rmsnorm_bwd(dx1n, x1, n2_w, rstd2, dx_add=d2)
        da = ops.gate_bwd(dx1, None, None, None)
        d_o = ops.gemm(da, w16(wo), b_mn=True)                                      # [R, D]
        del da
        if keep is not None:
            d_o.view(B, T, D).mul_(keep)
        q3 = qkv.view(B, T, 3 * D)
        dqkv = torch.empty_like(qkv)
        dq3 = dqkv.view(B, T, 3 * D)
        ops.attn_dense_bwd(q3[..., :D], q3[..., D:2 * D], q3[..., 2 * D:], o, d_o.view(B, T, D), lse, heads, hd, scale,
                           causal=mask is None, mask=mask, slopes=None, pure_causal_flag=pure_flag,
                           dq=dq3[..., :D], dk=dq3[..., D:2 * D], dv=dq3[..., 2 * D:])
        ops.rope_(dqkv, B, T, 2 * heads, hd, cos, sin, inverse=True)               # d(rotated) -> d(projection)
        dxn = ops.gemm(dqkv, wqkv, b_mn=True)
        dx = ops.rmsnorm_bwd(dxn, x2d, n1_w, rstd1, dx_add=dx1)
        return (dx.view(B, T, D),) + (None,) * 14


def llama_decline_reason(block, hidden_states, attention_mask=None, position_embeddings=None, past_key_values=None,
                         use_cache=False, output_attentions=False):
    """Why FastLlamaBlock must hand this call to HF's own LlamaDecoderLayer.forward, or None when the fast path
    applies.  Needs no GPU: every check reads shapes, dtypes, flags and the block's configuration."""
    a, m = block.self_attn, block.mlp
    cfg = a.config
    D = hidden_states.shape[-1]
    hd = a.head_dim
    if past_key_values is not None or use_cache:
        return "KV cache"
    if output_attentions:
        return "output_attentions"
    if any(p.requires_grad for p in block.parameters()):
        return "trainable block parameters (this path has no wgrad)"
    if block.training and a.attention_dropout > 0:
        return "attention dropout in training"
    if cfg.num_key_value_heads != cfg.num_attention_heads or a.num_key_value_groups != 1:
        return "grouped-query attention"
    if any(lin.bias is not None for lin in (a.q_proj, a.k_proj, a.v_proj, a.o_proj, m.gate_proj, m.up_proj, m.down_proj)):
        return "attention_bias / mlp_bias"
    if m.config.hidden_act != "silu":
        return f"hidden_act {m.config.hidden_act!r}"
    if hd not in (64, 128):
        return f"head_dim {hd}"
    if abs(a.scaling - hd ** -0.5) > 1e-9:
        return "attention scaling other than head_dim ** -0.5"
    if a.q_proj.out_features != D or D > 4096:
        return f"hidden size {D} (needs num_heads * head_dim == hidden_size <= 4096)"
    if m.gate_proj.out_features % L.SWIGLU_GROUP != 0:
        return f"intermediate_size not a multiple of {L.SWIGLU_GROUP}"
    if position_embeddings is None:
        return "no position_embeddings"
    cos, sin = position_embeddings
    if cos.shape[-1] != hd or sin.shape != cos.shape:
        return "partial rotary embedding"
    if cos.dtype != f32 or sin.dtype != f32:
        return "cos / sin not float32"
    if attention_mask is not None:
        am = attention_mask
        B, T = hidden_states.shape[0], hidden_states.shape[1]
        if am.dtype != torch.bool:
            return "float / additive attention mask"
        if am.dim() != 4 or am.shape[0] not in (1, B) or am.shape[1] != 1 or am.shape[2] != T or am.shape[3] != T:
            return "attention mask shape"
    if not hidden_states.is_cuda:
        return "not on CUDA"
    return None


class FastLlamaBlock:
    """Callable with HF LlamaDecoderLayer.forward's signature; returns None when the fast path does not apply."""

    def __init__(self, block):
        self.block = block
        self._packed = None   # (source-parameter versions and pointers, bf16 [q; k; v], bf16 packed [gate; up])

    def _weights(self):
        """Cached bf16 copies of the fused QKV and the packed gate/up weight, rebuilt when a source parameter
        changes (load_state_dict after construction, an in-place edit)."""
        a, m = self.block.self_attn, self.block.mlp
        src = (a.q_proj.weight, a.k_proj.weight, a.v_proj.weight, m.gate_proj.weight, m.up_proj.weight)
        key = tuple((p._version, p.data_ptr(), p.device) for p in src)
        if self._packed is None or self._packed[0] != key:
            with torch.no_grad():
                wqkv = torch.cat(src[:3], 0).to(bf16).contiguous()
                wgu = pack_gate_up(src[3], src[4]).to(bf16).contiguous()
            self._packed = (key, wqkv, wgu)
        return self._packed[1], self._packed[2]

    def __call__(self, hidden_states, attention_mask=None, position_ids=None, past_key_values=None, use_cache=False,
                 position_embeddings=None, pure_causal_flag=None, output_attentions=False, **kwargs):
        if not ENABLED or llama_decline_reason(self.block, hidden_states, attention_mask, position_embeddings,
                                               past_key_values, use_cache, output_attentions) is not None:
            return None
        b = self.block
        B, T, D = hidden_states.shape
        mask = keep = None
        if attention_mask is not None:
            m = attention_mask
            ref = _llama_mask_cache[0]
            if ref is not None and ref() is m and _llama_mask_cache[1].shape[0] == B:
                mask, keep = _llama_mask_cache[1], _llama_mask_cache[2]
            else:
                m = m.expand(B, 1, T, T).reshape(B, T, T)
                mask = (~m).contiguous()                                 # HF: True = attend; kernel: nonzero = masked
                keep = m.any(-1, keepdim=True).to(bf16)                 # 0 for a query with no allowed key
                _llama_mask_cache[0], _llama_mask_cache[1], _llama_mask_cache[2] = weakref.ref(attention_mask), mask, keep
        cos, sin = position_embeddings
        cos, sin = cos.contiguous(), sin.contiguous()
        wqkv, wgu = self._weights()
        a, mlp = b.self_attn, b.mlp
        x = hidden_states if hidden_states.dtype == f32 else hidden_states.float()
        out = FrozenLlamaBlockFn.apply(x, mask, keep, pure_causal_flag if mask is not None else None, cos, sin,
                                       a.config.num_attention_heads, b.input_layernorm.variance_epsilon,
                                       b.post_attention_layernorm.variance_epsilon, b.input_layernorm.weight, wqkv,
                                       a.o_proj.weight, b.post_attention_layernorm.weight, wgu, mlp.down_proj.weight)
        if out.dtype != hidden_states.dtype:
            out = out.to(hidden_states.dtype)
        return out


def accelerate(decoder_layer):
    """Return a fast evaluator for a recognised frozen decoder block, else None."""
    if type(decoder_layer).__name__ == "MptBlock" and hasattr(decoder_layer, "attn") and hasattr(decoder_layer, "ffn"):
        return FastMptBlock(decoder_layer)
    if type(decoder_layer).__name__ == "LlamaDecoderLayer" and hasattr(decoder_layer, "self_attn") and \
            hasattr(decoder_layer, "mlp"):
        return FastLlamaBlock(decoder_layer)
    return None
