"""Thin, shape-checked Python wrappers over the libofk.so C ABI (one function per entry point).

These do no math of their own.  Argument-shape violations raise ValueError/AssertionError *before* the
call (mirroring the reference's conventions, e.g. helpers.py:175-178); nonzero return codes from the
library become RuntimeError.
"""
import os

import torch

from . import _lib as L

bf16 = torch.bfloat16
f32 = torch.float32


def _rowmajor_2d(t, name):
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"{name} must be 2-D with unit inner stride, got shape {tuple(t.shape)} stride {t.stride()}")


_gemm_ws = {}


def _gemm_workspace(device):
    """Scratch for the GEMM tail split (see ofk_gemm_bf16_ws): one buffer per (device, stream) so GEMMs that may
    overlap never share it.  Allocated through torch's caching allocator, which is also legal while a CUDA graph
    is being captured (the buffer then lives in the graph's private pool and is kept alive here)."""
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ws = _gemm_ws.get(key)
    if ws is None:
        ws = torch.empty(int(L.lib().ofk_gemm_workspace_bytes()), device=device, dtype=torch.uint8)
        ws[:16384].zero_()   # the flag words (first 16 KiB); they reset themselves after every use
        _gemm_ws[key] = ws
    return ws


_comm_in_flight = False
# SMs every persistent GEMM grid leaves to NCCL while gradient-chunk all-reduces are in flight (world > 1 only; 0 = none).
# Measured at N = 2 inside the captured step (profiles/r02_ddp_timeline_n2.md): with all 148 SMs owned by the GEMM grids the
# all-reduce kernels are starved (30.8 ms of NCCL kernel time) and the ~60 GEMMs that run beside them take 1.3-1.55 x longer
# (static tile schedule: the clusters that cannot become resident do their share afterwards) -- 121.1 ms / step; with 16 SMs
# left free (and NCCL_MAX_CTAS=16, see train.configure_nccl_for_overlap) 117.7 ms.
COMM_RESERVED_SMS = int(os.environ.get("OFK_COMM_RESERVE_SMS", "16"))


def set_comm_in_flight(flag):
    """train.GradBucket brackets the window in which gradient-chunk all-reduces may be running.  Inside it (a) the GEMM
    tail split is not used: its owner slice spins on flags written by OTHER clusters of the same persistent grid,
    which assumes all clusters are co-resident -- not guaranteed while NCCL's CTAs hold SMs; (b) the persistent GEMM
    grids are shrunk by COMM_RESERVED_SMS so the collective's CTAs can run BESIDE the GEMMs instead of between them."""
    global _comm_in_flight
    flag = bool(flag)
    if flag != _comm_in_flight and COMM_RESERVED_SMS > 0:
        L.lib().ofk_gemm_reserve_sms(COMM_RESERVED_SMS if flag else 0)
    _comm_in_flight = flag


def gemm(a, b, *, a_mn=False, b_mn=False, epi=L.EPI_STORE_BF16, out=None, out2=None, aux=None, bias=None,
         gate=None, splits=1, block_n=0, M=None, N=None, K=None):
    """out[m,n] = epi(sum_k A(m,k) B(n,k)).

    a: [M,K] (a_mn=False) or [K,M] (a_mn=True); b: [N,K] (b_mn=False) or [K,N] (b_mn=True); both bf16.
    """
    L.require_cuda(a, b)
    _rowmajor_2d(a, "a")
    _rowmajor_2d(b, "b")
    if a.dtype != bf16 or b.dtype != bf16:
        raise ValueError("gemm operands must be bfloat16")
    m, ka = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
    n, kb = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
    if ka != kb:
        raise ValueError(f"gemm reduction dims differ: {ka} vs {kb}")
    M = m if M is None else M
    N = n if N is None else N
    K = ka if K is None else K
    out_dtype = f32 if epi in (L.EPI_STORE_F32, L.EPI_ATOMIC_F32, L.EPI_GATE_RESID_F32,
                               L.EPI_BIAS_RESID_F32) else bf16
    if out is None:
        if epi == L.EPI_ATOMIC_F32:
            raise ValueError("atomic epilogue accumulates into an existing `out`")
        out = torch.empty((M, N), device=a.device, dtype=out_dtype)
    _rowmajor_2d(out, "out")
    if out.dtype != out_dtype or out.shape[0] < M or out.shape[1] < N:
        raise ValueError(f"bad out tensor {tuple(out.shape)} {out.dtype} for ({M},{N}) {out_dtype}")
    if out2 is not None:
        _rowmajor_2d(out2, "out2")
    if aux is not None:
        _rowmajor_2d(aux, "aux")
    if bias is not None and (bias.dtype != f32 or bias.numel() < N or not bias.is_contiguous()):
        raise ValueError("gemm bias must be a contiguous float32 vector of length >= N")
    if gate is not None and gate.dtype != f32:
        raise ValueError("gemm gate must be float32")
    ws = _gemm_workspace(a.device) if (splits == 1 and M >= 512 and N >= 256 and K >= 3072 and not _comm_in_flight) \
        else None
    L.check(L.lib().ofk_gemm_bf16_ws(
        epi, int(a_mn), int(b_mn), a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), M, N, K, splits, block_n,
        out.data_ptr(), out.stride(0), L.ptr(out2), 0 if out2 is None else out2.stride(0),
        L.ptr(aux), 0 if aux is None else aux.stride(0), L.ptr(bias), L.ptr(gate),
        L.ptr(ws), 0 if ws is None else ws.numel(), L.stream_ptr()))
    return out


def layernorm_fwd(x, gamma, beta, eps=1e-5, *, out=None, out_f32=False, rows_per_group=0, group_stride=0,
                  group_offset=0, want_stats=True):
    """x: [rows, D] f32.  Returns (y, mean, rstd).  `out` may be a larger buffer written with the group mapping."""
    L.require_cuda(x)
    _rowmajor_2d(x, "x")
    if x.dtype != f32:
        raise ValueError("layernorm input must be float32 (the residual stream is fp32)")
    rows, D = x.shape
    if out is None:
        out = torch.empty((rows, D), device=x.device, dtype=f32 if out_f32 else bf16)
    _rowmajor_2d(out, "out")
    y_is_f32 = out.dtype == f32
    mean = torch.empty(rows, device=x.device, dtype=f32) if want_stats else None
    rstd = torch.empty(rows, device=x.device, dtype=f32) if want_stats else None
    L.check(L.lib().ofk_layernorm_fwd(x.data_ptr(), x.stride(0), gamma.data_ptr(), beta.data_ptr(), eps, rows, D,
                                      out.data_ptr(), int(y_is_f32), out.stride(0), rows_per_group, group_stride,
                                      group_offset, L.ptr(mean), L.ptr(rstd), L.stream_ptr()))
    return out, mean, rstd


_ln_ws = {}


def _ln_workspace(device, rows, D):
    need = int(L.lib().ofk_layernorm_bwd_workspace(rows, D))
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _ln_ws.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, device=device, dtype=torch.uint8)
        _ln_ws[key] = ws
    return ws


def layernorm_bwd(dy, x, gamma, mean, rstd, *, dgamma=None, dbeta=None, dx=None, dx_add=None, rows_per_group=0,
                  group_stride=0, group_offset=0, want_dx=True):
    """dx = LN'(dy) (+ dx_add); dgamma/dbeta are accumulated in place.  dy may be bf16 or f32 (mapped rows).
    want_dx=False: only the affine-parameter gradients are produced."""
    L.require_cuda(dy, x)
    _rowmajor_2d(dy, "dy")
    _rowmajor_2d(x, "x")
    rows, D = x.shape
    if dx is None and want_dx:
        dx = torch.empty((rows, D), device=x.device, dtype=f32)
    ws = _ln_workspace(x.device, rows, D)
    L.check(L.lib().ofk_layernorm_bwd(dy.data_ptr(), int(dy.dtype == f32), dy.stride(0), rows_per_group, group_stride,
                                      group_offset, x.data_ptr(), x.stride(0), gamma.data_ptr(), mean.data_ptr(),
                                      rstd.data_ptr(), rows, D, L.ptr(dx), 0 if dx is None else dx.stride(0), L.ptr(dx_add),
                                      0 if dx_add is None else dx_add.stride(0), L.ptr(dgamma), L.ptr(dbeta),
                                      ws.data_ptr(), L.stream_ptr()))
    return dx


def _bstride_ld(t, name):
    if t.dim() != 3 or t.stride(2) != 1:
        raise ValueError(f"{name} must be [batch, rows, heads*64] with unit inner stride")
    return t.stride(0), t.stride(1)


def attn_force_legacy(on):
    """A/B switch: True = always the mma.sync attention kernels, False = TMA + tcgen05 whenever the layout allows
    (the default).  Returns the previous setting."""
    return bool(L.lib().ofk_attn_force_legacy(int(bool(on))))


def attn_tc_launch_count():
    return int(L.lib().ofk_attn_tc_launch_count())


_attn_ws = {}


def _attn_workspace(device, nbytes):
    """fp32 dQ accumulator of the tensor-core attention backward (one per (device, stream), grown on demand)."""
    if nbytes <= 0:
        return None
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ws = _attn_ws.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes), device=device, dtype=torch.uint8)
        _attn_ws[key] = ws
    return ws


def attn_fwd(q, k, v, heads, scale, *, mask_mode=L.MASK_NONE, text_time=None, keys_per_media=64, out=None,
             want_lse=True):
    """q: [B, nq, heads*64] (may be a column-slice view), k/v: [B, nk, heads*64].  Returns (o, lse)."""
    L.require_cuda(q, k, v)
    B, nq = q.shape[0], q.shape[1]
    nk = k.shape[1]
    if q.dtype != bf16 or k.dtype != bf16 or v.dtype != bf16:
        raise ValueError("attention operands must be bfloat16")
    if out is None:
        out = torch.empty((B, nq, heads * 64), device=q.device, dtype=bf16)
    lse = torch.empty((B, heads, nq), device=q.device, dtype=f32) if want_lse else None
    qb, ldq = _bstride_ld(q, "q")
    kb, ldk = _bstride_ld(k, "k")
    vb, ldv = _bstride_ld(v, "v")
    ob, ldo = _bstride_ld(out, "out")
    if mask_mode != L.MASK_NONE:
        if text_time is None or text_time.dtype != torch.int32 or tuple(text_time.shape) != (B, nq):
            raise ValueError("media mask needs int32 text_time of shape [B, nq]")
        text_time = text_time.contiguous()
    L.check(L.lib().ofk_attn_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), L.ptr(lse), B, heads, nq, nk,
                                 qb, ldq, kb, ldk, vb, ldv, ob, ldo, scale, mask_mode, L.ptr(text_time), keys_per_media,
                                 L.stream_ptr()))
    return out, lse


def attn_bwd(q, k, v, o, d_o, lse, heads, scale, *, mask_mode=L.MASK_NONE, text_time=None, keys_per_media=64,
             dq=None, dk=None, dv=None):
    """Returns (dq, dk, dv) bf16.  d_o must share o's strides."""
    L.require_cuda(q, k, v, o, d_o)
    B, nq = q.shape[0], q.shape[1]
    nk = k.shape[1]
    if d_o.stride() != o.stride():
        raise ValueError("d_o must have the same strides as o")
    if dq is None:
        dq = torch.empty((B, nq, heads * 64), device=q.device, dtype=bf16)
    if dk is None:
        dk = torch.empty((B, nk, heads * 64), device=q.device, dtype=bf16)
    if dv is None:
        dv = torch.empty((B, nk, heads * 64), device=q.device, dtype=bf16)
    delta = torch.empty((B, heads, nq), device=q.device, dtype=f32)
    qb, ldq = _bstride_ld(q, "q")
    kb, ldk = _bstride_ld(k, "k")
    vb, ldv = _bstride_ld(v, "v")
    ob, ldo = _bstride_ld(o, "o")
    dqb, lddq = _bstride_ld(dq, "dq")
    dkb, lddk = _bstride_ld(dk, "dk")
    dvb, lddv = _bstride_ld(dv, "dv")
    if text_time is not None:
        text_time = text_time.contiguous()
    ws = _attn_workspace(q.device, L.lib().ofk_attn_bwd_workspace_bytes(B, heads, 64, nq, nk))
    L.check(L.lib().ofk_attn_bwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), d_o.data_ptr(), lse.data_ptr(),
                                 delta.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), B, heads, nq, nk,
                                 qb, ldq, kb, ldk, vb, ldv, ob, ldo, dqb, lddq, dkb, lddk, dvb, lddv, scale, mask_mode,
                                 L.ptr(text_time), keys_per_media, L.ptr(ws), 0 if ws is None else ws.numel(),
                                 L.stream_ptr()))
    return dq, dk, dv


def make_labels(input_ids, pad_token_id, media_token_id, endofchunk_token_id=None, interleaved=False, out=None):
    """Device-side training labels (train_utils.py:102-106; interleaved=True: the MMC4 rule of :126-149).
    input_ids: int64 [B, T] on the GPU (row stride free).  Returns int64 [B, T]."""
    L.require_cuda(input_ids)
    if input_ids.dtype != torch.int64 or input_ids.dim() != 2 or (input_ids.numel() and input_ids.stride(1) != 1):
        raise ValueError("make_labels expects an int64 [B, T] tensor with contiguous rows")
    if interleaved and endofchunk_token_id is None:
        raise ValueError("interleaved labels need the <|endofchunk|> token id")
    B, T = input_ids.shape
    if out is None:
        out = torch.empty((B, T), device=input_ids.device, dtype=torch.int64)
    if B == 0 or T == 0:
        return out
    L.check(L.lib().ofk_make_labels(input_ids.data_ptr(), input_ids.stride(0), B, T, int(pad_token_id),
                                    int(media_token_id), int(-1 if endofchunk_token_id is None else endofchunk_token_id),
                                    int(bool(interleaved)), out.data_ptr(), out.stride(0), L.stream_ptr()))
    return out


def text_time(input_ids=None, media_token_id=0, media_locations=None, use_cached_media=False, t_txt=None):
    """int32 [B, T_txt] inclusive count of media tokens (helpers.py:199-208)."""
    src = media_locations if media_locations is not None else input_ids
    L.require_cuda(src)
    B = src.shape[0]
    n_loc = src.shape[1]
    if t_txt is None:
        t_txt = n_loc
    loc = None
    if media_locations is not None:
        loc = media_locations.to(torch.uint8).contiguous()
    ids = None
    if input_ids is not None and media_locations is None:
        ids = input_ids.to(torch.int64).contiguous()
    out = torch.empty((B, t_txt), device=src.device, dtype=torch.int32)
    L.check(L.lib().ofk_text_time(L.ptr(ids), int(media_token_id), B, t_txt, n_loc, L.ptr(loc), int(use_cached_media),
                                  out.data_ptr(), L.stream_ptr()))
    return out


def cast_bf16(src, out=None):
    L.require_cuda(src)
    src = src.contiguous()
    if out is None:
        out = torch.empty(src.shape, device=src.device, dtype=bf16)
    L.check(L.lib().ofk_cast_f32_bf16(src.data_ptr(), out.data_ptr(), src.numel(), L.stream_ptr()))
    return out


def gate_bwd(dout, branch, gate, dgate):
    """dbranch(bf16) = dout * tanh(gate); dgate += (1 - tanh^2) * <dout, branch>.  gate None: plain cast."""
    L.require_cuda(dout)
    if not dout.is_contiguous() or (branch is not None and not branch.is_contiguous()):
        raise ValueError("gate_bwd operands must be contiguous")
    dbranch = torch.empty(dout.shape, device=dout.device, dtype=bf16)
    L.check(L.lib().ofk_gate_bwd(dout.data_ptr(), L.ptr(branch), L.ptr(gate), dbranch.data_ptr(), L.ptr(dgate),
                                 dout.numel(), L.stream_ptr()))
    return dbranch


def add_(dst, src):
    L.check(L.lib().ofk_add_f32(dst.data_ptr(), src.data_ptr(), dst.numel(), L.stream_ptr()))
    return dst


def patchify(images, patch, ldp):
    """images [n,3,H,W] f32 -> [n*g, ldp] bf16 patch rows (conv-weight column order), zero padded."""
    L.require_cuda(images)
    images = images.contiguous()
    n, _, H, W = images.shape
    g = (H // patch) * (W // patch)
    out = torch.empty((n * g, ldp), device=images.device, dtype=bf16)
    L.check(L.lib().ofk_patchify(images.data_ptr(), n, H, W, patch, out.data_ptr(), ldp, L.stream_ptr()))
    return out


def vit_assemble(patch_emb, class_emb, pos_emb, n, g, D):
    tok = torch.empty((n * (g + 1), D), device=patch_emb.device, dtype=f32)
    L.check(L.lib().ofk_vit_assemble(patch_emb.data_ptr(), class_emb.data_ptr(), pos_emb.data_ptr(), n, g, D,
                                     tok.data_ptr(), L.stream_ptr()))
    return tok


def adamw_(param, grad, exp_avg, exp_avg_sq, w_bf16, lr, beta1, beta2, eps, wd, step, clip_scale=None, step_dev=None,
           lr_dev=None):
    """step: host int (ignored when step_dev, a device float tensor holding the step count, is given)."""
    bc1 = 1.0 - beta1 ** max(step, 1)
    bc2 = 1.0 - beta2 ** max(step, 1)
    L.check(L.lib().ofk_adamw(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                              L.ptr(w_bf16), param.numel(), lr, beta1, beta2, eps, wd, bc1, bc2, L.ptr(clip_scale),
                              L.ptr(step_dev), L.ptr(lr_dev), L.stream_ptr()))


def sumsq_(x, out):
    L.check(L.lib().ofk_sumsq(x.data_ptr(), x.numel(), out.data_ptr(), L.stream_ptr()))
    return out


def attn_dense_fwd(q, k, v, heads, head_dim, scale, *, causal=False, mask=None, slopes=None, pure_causal_flag=None,
                   want_lse=True):
    """Dense (LM self-attention) core: q/k/v [B, n, heads*head_dim] strided views; mask [B, nq, nk] bool/uint8
    (True = masked); slopes [heads] f32 ALiBi slopes.  Returns (o, lse)."""
    L.require_cuda(q, k, v)
    B, nq, nk = q.shape[0], q.shape[1], k.shape[1]
    out = torch.empty((B, nq, heads * head_dim), device=q.device, dtype=bf16)
    lse = torch.empty((B, heads, nq), device=q.device, dtype=f32) if want_lse else None
    qb, ldq = _bstride_ld(q, "q")
    kb, ldk = _bstride_ld(k, "k")
    vb, ldv = _bstride_ld(v, "v")
    ob, ldo = _bstride_ld(out, "out")
    if mask is not None and (tuple(mask.shape) != (B, nq, nk) or not mask.is_contiguous() or mask.element_size() != 1):
        raise ValueError("mask must be a contiguous 1-byte tensor of shape [B, nq, nk]")
    L.check(L.lib().ofk_attn_dense_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), L.ptr(lse), B, heads,
                                       head_dim, nq, nk, qb, ldq, kb, ldk, vb, ldv, ob, ldo, scale, int(causal),
                                       L.ptr(mask), L.ptr(slopes), L.ptr(pure_causal_flag), L.stream_ptr()))
    return out, lse


def attn_dense_bwd(q, k, v, o, d_o, lse, heads, head_dim, scale, *, causal=False, mask=None, slopes=None,
                   pure_causal_flag=None, dq=None, dk=None, dv=None):
    L.require_cuda(q, k, v, o, d_o)
    B, nq, nk = q.shape[0], q.shape[1], k.shape[1]
    if d_o.stride() != o.stride():
        raise ValueError("d_o must have the same strides as o")
    inner = heads * head_dim
    if dq is None:
        dq = torch.empty((B, nq, inner), device=q.device, dtype=bf16)
    if dk is None:
        dk = torch.empty((B, nk, inner), device=q.device, dtype=bf16)
    if dv is None:
        dv = torch.empty((B, nk, inner), device=q.device, dtype=bf16)
    delta = torch.empty((B, heads, nq), device=q.device, dtype=f32)
    qb, ldq = _bstride_ld(q, "q")
    kb, ldk = _bstride_ld(k, "k")
    vb, ldv = _bstride_ld(v, "v")
    ob, ldo = _bstride_ld(o, "o")
    dqb, lddq = _bstride_ld(dq, "dq")
    dkb, lddk = _bstride_ld(dk, "dk")
    dvb, lddv = _bstride_ld(dv, "dv")
    ws = _attn_workspace(q.device, L.lib().ofk_attn_bwd_workspace_bytes(B, heads, head_dim, nq, nk))
    L.check(L.lib().ofk_attn_dense_bwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), d_o.data_ptr(),
                                       lse.data_ptr(), delta.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(),
                                       B, heads, head_dim, nq, nk, qb, ldq, kb, ldk, vb, ldv, ob, ldo, dqb, lddq, dkb,
                                       lddk, dvb, lddv, scale, int(causal), L.ptr(mask), L.ptr(slopes),
                                       L.ptr(pure_causal_flag), L.ptr(ws), 0 if ws is None else ws.numel(),
                                       L.stream_ptr()))
    return dq, dk, dv


def gemm_grouped(a, b, *, a_mn=False, b_mn=False, epi=L.EPI_STORE_BF16, out, M, N, K, bias=None, splits=1, block_n=0,
                 out_map=(0, 0, 0), ak_map=(0, 0, 0)):
    """GEMM with grouped row maps (see ofk_gemm_bf16_grouped): `out_map` = (rows_per_group, group_stride,
    group_offset) for the rows of `out`; `ak_map` the same for the reduction rows of an MN-major `a`."""
    L.require_cuda(a, b, out)
    _rowmajor_2d(a, "a")
    _rowmajor_2d(b, "b")
    _rowmajor_2d(out, "out")
    if a.dtype != bf16 or b.dtype != bf16:
        raise ValueError("gemm operands must be bfloat16")
    if bias is not None and (bias.dtype != f32 or bias.numel() < N or not bias.is_contiguous()):
        raise ValueError("gemm bias must be a contiguous float32 vector of length >= N")
    L.check(L.lib().ofk_gemm_bf16_grouped(
        epi, int(a_mn), int(b_mn), a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), M, N, K, splits, block_n,
        out.data_ptr(), out.stride(0), L.ptr(bias), out_map[0], out_map[1], out_map[2], ak_map[0], ak_map[1], ak_map[2],
        L.stream_ptr()))
    return out


def rmsnorm_fwd(x, gamma, eps):
    """x: [rows, D] f32.  Returns (y bf16, rstd f32 [rows])."""
    L.require_cuda(x, gamma)
    _rowmajor_2d(x, "x")
    if x.dtype != f32 or gamma.dtype != f32 or not gamma.is_contiguous() or gamma.numel() != x.shape[1]:
        raise ValueError("rmsnorm expects float32 x [rows, D] and a contiguous float32 gamma [D]")
    rows, D = x.shape
    y = torch.empty((rows, D), device=x.device, dtype=bf16)
    rstd = torch.empty(rows, device=x.device, dtype=f32)
    L.check(L.lib().ofk_rmsnorm_fwd(x.data_ptr(), x.stride(0), gamma.data_ptr(), eps, rows, D, y.data_ptr(), y.stride(0),
                                    rstd.data_ptr(), L.stream_ptr()))
    return y, rstd


def rmsnorm_bwd(dy, x, gamma, rstd, *, dx_add=None):
    """dx(f32) = RMSNorm'(dy) (+ dx_add).  dy bf16 or f32 [rows, D]; gamma frozen (no dgamma)."""
    L.require_cuda(dy, x, gamma, rstd, dx_add)
    _rowmajor_2d(dy, "dy")
    _rowmajor_2d(x, "x")
    if dy.shape != x.shape or x.dtype != f32 or dy.dtype not in (bf16, f32):
        raise ValueError("rmsnorm_bwd: dy (bf16/f32) and x (f32) must share the shape [rows, D]")
    if dx_add is not None:
        _rowmajor_2d(dx_add, "dx_add")
        if dx_add.dtype != f32 or dx_add.shape != x.shape:
            raise ValueError("rmsnorm_bwd: dx_add must be float32 like x")
    rows, D = x.shape
    dx = torch.empty((rows, D), device=x.device, dtype=f32)
    L.check(L.lib().ofk_rmsnorm_bwd(dy.data_ptr(), int(dy.dtype == f32), dy.stride(0), x.data_ptr(), x.stride(0),
                                    gamma.data_ptr(), rstd.data_ptr(), rows, D, dx.data_ptr(), dx.stride(0),
                                    L.ptr(dx_add), 0 if dx_add is None else dx_add.stride(0), L.stream_ptr()))
    return dx


def rope_(x, batch, T, nheads, head_dim, cos, sin, *, inverse=False):
    """In place on x [batch*T, ld] bf16: rotate the first nheads heads of every row (HF apply_rotary_pos_emb;
    inverse=True applies its transpose, for the backward).  cos / sin: f32 [1 or batch, T, head_dim]."""
    L.require_cuda(x, cos, sin)
    _rowmajor_2d(x, "x")
    if x.dtype != bf16 or x.shape[0] != batch * T or x.shape[1] < nheads * head_dim:
        raise ValueError(f"rope: x must be bf16 [{batch * T}, >= {nheads * head_dim}], got {tuple(x.shape)} {x.dtype}")
    for t, name in ((cos, "cos"), (sin, "sin")):
        if t.dtype != f32 or t.dim() != 3 or t.shape[0] not in (1, batch) or tuple(t.shape[1:]) != (T, head_dim) \
                or not t.is_contiguous():
            raise ValueError(f"rope: {name} must be a contiguous float32 [1 or {batch}, {T}, {head_dim}] tensor")
    if cos.shape != sin.shape:
        raise ValueError("rope: cos and sin shapes differ")
    cs_bstride = 0 if cos.shape[0] == 1 else T * head_dim
    L.check(L.lib().ofk_rope(x.data_ptr(), x.stride(0), batch, T, nheads, head_dim, cos.data_ptr(), sin.data_ptr(),
                             cs_bstride, int(bool(inverse)), L.stream_ptr()))
    return x


def swiglu_gemm(x, w_packed, *, want_gu=True):
    """h = bf16(silu(g)) * u for the packed [gate; up] weight (OFK_EPI_SWIGLU_DUAL).  x: [R, D] bf16,
    w_packed: [2I, D] bf16.  Returns (h [R, I], gu [R, 2I] packed raw projections or None)."""
    L.require_cuda(x, w_packed)
    _rowmajor_2d(x, "x")
    _rowmajor_2d(w_packed, "w_packed")
    if x.dtype != bf16 or w_packed.dtype != bf16:
        raise ValueError("swiglu_gemm operands must be bfloat16")
    R, K = x.shape
    N = w_packed.shape[0]
    if w_packed.shape[1] != K or N % (2 * L.SWIGLU_GROUP) != 0:
        raise ValueError(f"swiglu_gemm: w_packed must be [2I, {K}] with I % {L.SWIGLU_GROUP} == 0, got {tuple(w_packed.shape)}")
    h = torch.empty((R, N // 2), device=x.device, dtype=bf16)
    gu = torch.empty((R, N), device=x.device, dtype=bf16) if want_gu else None
    ws = _gemm_workspace(x.device) if (R >= 512 and N >= 256 and K >= 3072 and not _comm_in_flight) else None
    L.check(L.lib().ofk_gemm_bf16_ws(
        L.EPI_SWIGLU_DUAL, 0, 0, x.data_ptr(), x.stride(0), w_packed.data_ptr(), w_packed.stride(0), R, N, K, 1, 0,
        h.data_ptr(), h.stride(0), L.ptr(gu), 0 if gu is None else gu.stride(0), 0, 0, 0, 0,
        L.ptr(ws), 0 if ws is None else ws.numel(), L.stream_ptr()))
    return h, gu


def swiglu_bwd(dh, gu):
    """dh: [R, I] bf16, gu: [R, 2I] packed bf16 g / u.  Returns dgu [R, 2I] bf16 in the packed order."""
    L.require_cuda(dh, gu)
    _rowmajor_2d(dh, "dh")
    _rowmajor_2d(gu, "gu")
    R, I = dh.shape
    if dh.dtype != bf16 or gu.dtype != bf16 or tuple(gu.shape) != (R, 2 * I):
        raise ValueError("swiglu_bwd: dh [R, I] and gu [R, 2I] must be bfloat16")
    dgu = torch.empty((R, 2 * I), device=dh.device, dtype=bf16)
    L.check(L.lib().ofk_swiglu_bwd(dh.data_ptr(), dh.stride(0), gu.data_ptr(), gu.stride(0), R, I, dgu.data_ptr(),
                                   dgu.stride(0), L.stream_ptr()))
    return dgu
