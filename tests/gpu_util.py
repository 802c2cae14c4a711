"""Helpers shared by the GPU parity tests: drive single kernels of libttsb.so through the C ABI."""
from __future__ import annotations

import numpy as np
import torch

from transformertts_b200 import lib
from transformertts_b200.model.models import _PackedLinear, _round_up

DEV = 'cuda:0'


def split_or_none(x: torch.Tensor, split: bool):
    return lib.split_bf16(x, split)


def dropout_keep_host(idx, p, seed, site, salt=0):
    """Host restatement of the library's stateless dropout mask (csrc/ttsb_common.cuh: dropout_keep): True where element
    `idx` (any integer array) of dropout site `site` is kept at rate p (float32, as the kernels receive it)."""
    idx = np.asarray(idx, dtype=np.uint64)
    pair = idx >> np.uint64(1)
    u32 = lambda v: np.uint32(int(v) & 0xffffffff)
    hterm = ((pair >> np.uint64(32)).astype(np.uint32) * u32(0x85EBCA77)) ^ u32(((seed ^ salt) & 0xffffffff) * 0xC2B2AE3D) \
        ^ u32(site * 0x27D4EB2F)
    x = (pair & np.uint64(0xffffffff)).astype(np.uint32) * u32(0x9E3779B1) ^ hterm
    x ^= x >> np.uint32(16)
    x *= u32(0x7FEB352D)
    x ^= x >> np.uint32(15)
    x *= u32(0x846CA68B)
    x ^= x >> np.uint32(16)
    half = np.where((idx & np.uint64(1)) != 0, x >> np.uint32(16), x & np.uint32(0xffff))
    thresh = int(float(np.float32(p)) * 4294967296.0) if p > 0 else 0
    return half >= np.uint32(thresh >> 16)


def run_gemm(x_list, w_kn, bias, seg_src, seg_shift, seg_k, *, precision='bf16x3', impl='tcgen05', relu=False,
             residual=None, ln=None, row_len=None, block_n=None, single_tile=False, out_fp16=False, drop_pre=None,
             drop_post=None, drop_seed=0, out_preln=False, want_f32=True):
    """x_list: fp32 (B,T,C) sources (on GPU).  Returns dict with requested outputs.  drop_pre / drop_post: (rate, site) of
    the two dropout sites of the epilogue; out_preln=True also returns the saved pre-LayerNorm values ('preln');
    want_f32=False leaves out_f32 NULL (16-bit outputs only).  'launches' counts the kernels ttsb_linear_fwd launched."""
    split = precision == 'bf16x3'
    B, T, _ = x_list[0].shape
    pl = _PackedLinear(w_kn, bias, seg_k, split, single_tile=single_tile, block_n=block_n)
    a = lib.GemmArgs()
    a.B, a.T, a.N, a.block_n = B, T, pl.N, pl.block_n
    a.num_segments = len(seg_k)
    keep = []
    for s in range(len(seg_k)):
        a.seg_src[s], a.seg_shift[s], a.seg_k[s] = seg_src[s], seg_shift[s], seg_k[s]
    for i, x in enumerate(x_list):
        hi, lo = lib.split_bf16(x, split)
        keep += [hi, lo]
        a.a_hi[i] = hi.data_ptr()
        a.a_lo[i] = lo.data_ptr() if lo is not None else None
        a.lda[i] = x.shape[-1]
        a.a_col0[i] = 0
    a.w_hi = pl.w_hi.data_ptr()
    a.w_lo = pl.w_lo.data_ptr() if pl.w_lo is not None else None
    a.bias = pl.bias.data_ptr() if pl.bias is not None else None
    a.relu = int(relu)
    if residual is not None:
        a.residual = residual.data_ptr()
        a.ld_res = residual.shape[-1]
    if ln is not None:
        from transformertts_b200.model.models import _pad_vec
        g_pad, b_pad = _pad_vec(ln[0], pl.n_pad), _pad_vec(ln[1], pl.n_pad)
        keep += [g_pad, b_pad]
        a.ln_gamma, a.ln_beta, a.ln_eps = g_pad.data_ptr(), b_pad.data_ptr(), 1e-6
    if row_len is not None:
        a.row_len = row_len.data_ptr()
    out = {}
    # poison the outputs so unwritten elements are visible
    out_f32 = torch.full((B, T, pl.n_pad), float('nan'), device=DEV)
    out_hi = torch.full((B, T, pl.n_pad), float('nan'), device=DEV, dtype=torch.bfloat16)
    out_lo = torch.full((B, T, pl.n_pad), float('nan'), device=DEV, dtype=torch.bfloat16)
    a.out_f32, a.out_hi = (out_f32.data_ptr() if want_f32 else None), out_hi.data_ptr()
    a.out_lo = out_lo.data_ptr() if split else None
    a.ld_out = pl.n_pad
    a.out_fp16 = int(out_fp16)
    preln = None
    if out_preln:
        preln = torch.full((B, T, pl.n_pad), float('nan'), device=DEV)
        a.out_preln = preln.data_ptr()
    if drop_pre is not None:
        a.drop_pre_p, a.drop_pre_site = drop_pre
    if drop_post is not None:
        a.drop_post_p, a.drop_post_site = drop_post
    a.drop_seed = drop_seed
    a.precision = lib.PREC_BF16X3 if split else lib.PREC_BF16
    a.impl = lib.IMPL_SIMT if impl == 'simt' else lib.IMPL_TCGEN05
    n0 = lib.launch_count()
    lib.linear_fwd(a)
    out['launches'] = lib.launch_count() - n0
    torch.cuda.synchronize()
    out['f32'] = out_f32 if want_f32 else None
    out['hi'] = out_hi
    out['lo'] = out_lo if split else None
    out['n_pad'] = pl.n_pad
    out['preln'] = preln
    return out


def ref_gemm(x_list, w_kn, bias, seg_src, seg_shift, seg_k, *, precision, relu=False, residual=None, ln=None, row_len=None,
             drop_pre=None, drop_post=None, drop_seed=0, salt=0, ld_out=None, return_preln=False):
    """float64 CPU reference of the same contract.  In 'bf16' mode the operands are first rounded to bf16 (that is the
    kernel's arithmetic); in 'bf16x3' mode the fp32 operands are used as they are.  Dropout uses the host mask at element
    index (b*T + t)*ld_out + n; return_preln=True returns (output, pre-LayerNorm value)."""
    xs = [x.detach().cpu().double() if precision == 'bf16x3' else x.detach().cpu().bfloat16().double() for x in x_list]
    w = w_kn.detach().cpu().reshape(-1, w_kn.shape[-1])
    w = w.double() if precision == 'bf16x3' else w.bfloat16().double()
    B, T, _ = xs[0].shape
    N = w.shape[1]
    acc = torch.zeros(B, T, N, dtype=torch.float64)
    koff = 0
    for s, k in enumerate(seg_k):
        x = xs[seg_src[s]]
        sh = seg_shift[s]
        lo, hi = max(0, -sh), min(T, T - sh)
        if hi > lo:
            acc[:, lo:hi] += x[:, lo + sh:hi + sh, :k] @ w[koff:koff + k]
        koff += k
    if bias is not None:
        acc += bias.detach().cpu().double()
    if relu:
        acc = torch.relu(acc)

    def drop(v, rate_site):
        rate, site = rate_site
        idx = (np.arange(B * T, dtype=np.uint64)[:, None] * np.uint64(ld_out) + np.arange(N, dtype=np.uint64)[None, :])
        keep = torch.from_numpy(dropout_keep_host(idx, rate, drop_seed, site, salt)).view(B, T, N)
        return v * keep / (1.0 - float(np.float32(rate)))

    if drop_pre is not None and drop_pre[0] > 0:
        acc = drop(acc, drop_pre)
    if residual is not None:
        acc += residual.detach().cpu().double()[..., :N]
    preln = acc.clone()
    if ln is not None:
        g, b = ln[0].detach().cpu().double(), ln[1].detach().cpu().double()
        mean = acc.mean(-1, keepdim=True)
        var = ((acc - mean) ** 2).mean(-1, keepdim=True)
        acc = (acc - mean) * torch.rsqrt(var + 1e-6) * g + b
    if drop_post is not None and drop_post[0] > 0:
        acc = drop(acc, drop_post)
    if row_len is not None:
        keep = torch.arange(T)[None, :] < row_len.detach().cpu()[:, None]
        acc = acc * keep[..., None]
    return (acc, preln) if return_preln else acc


def _to16(x, precision, split):
    if precision == 'fp16':
        return x.contiguous().half(), None
    return lib.split_bf16(x, split)


def run_mha(q, k, v, kv_len, H, *, precision='bf16x3', impl='tcgen05', weights_b=None):
    """q,k,v fp32 (B,T,d) on GPU -> attention output fp32 (B,T,d) (hi+lo recombined)."""
    split = precision == 'bf16x3'
    B, T, d = q.shape
    dh = d // H
    qk = torch.cat([q, k, v], dim=-1).contiguous()
    qk_hi, qk_lo = _to16(qk, precision, split)
    out_hi = torch.full((B, T, d), float('nan'), device=DEV, dtype=torch.bfloat16)
    out_lo = torch.full((B, T, d), float('nan'), device=DEV, dtype=torch.bfloat16)
    m = lib.MhaArgs()
    m.B, m.T, m.H, m.dh = B, T, H, dh
    m.qk_hi = qk_hi.data_ptr()
    m.qk_lo = qk_lo.data_ptr() if split else None
    m.ld_qk, m.q_col0, m.k_col0, m.v_col0 = 3 * d, 0, d, 2 * d
    m.kv_len = kv_len.data_ptr()
    m.out_hi = out_hi.data_ptr()
    m.out_lo = out_lo.data_ptr()
    m.ld_out = d
    wts = None
    if weights_b is not None:
        wts = torch.full((H, T, T), float('nan'), device=DEV)
        m.weights_out = wts.data_ptr()
        m.weights_batch_index = weights_b
    m.precision = {'bf16x3': lib.PREC_BF16X3, 'bf16': lib.PREC_BF16, 'fp16': lib.PREC_FP16}[precision]
    m.impl = lib.IMPL_SIMT if impl == 'simt' else lib.IMPL_TCGEN05
    lib.mha_fwd(m)
    torch.cuda.synchronize()
    out = out_hi.float() + out_lo.float()
    return out, wts


def ref_mha(q, k, v, kv_len, H, precision):
    """float64 CPU attention with the reference's additive -1e9 key mask (model/layers.py:176-195)."""
    cast = {'bf16x3': lambda t: t.detach().cpu().double(), 'bf16': lambda t: t.detach().cpu().bfloat16().double(),
            'fp16': lambda t: t.detach().cpu().half().double()}[precision]
    q, k, v = cast(q), cast(k), cast(v)
    B, T, d = q.shape
    dh = d // H
    sp = lambda t: t.reshape(B, T, H, dh).permute(0, 2, 1, 3)
    logits = sp(q) @ sp(k).transpose(-1, -2) / (dh ** 0.5)
    mask = (torch.arange(T)[None, :] >= kv_len.cpu()[:, None]).double()[:, None, None, :]
    logits = (logits.float() + (mask * -1e9).float()).double()  # fp32 add as in the reference
    w = torch.softmax(logits, -1)
    out = (w @ sp(v)).permute(0, 2, 1, 3).reshape(B, T, d)
    return out, w


def run_mha_general(q, kv_k, kv_v, kv_len, H, *, precision='fp16', impl='tcgen05', causal=False, cross=False, full_queries=True,
                    weights_all=False):
    """General form of ttsb_mha_fwd: q fp32 (B,T,d); k,v fp32 (B,Tk,d).  cross=True keeps k|v in a second buffer."""
    split = precision == 'bf16x3'
    B, T, d = q.shape
    Tk = kv_k.shape[1]
    dh = d // H
    m = lib.MhaArgs()
    m.B, m.T, m.H, m.dh = B, T, H, dh
    if cross:
        qb_hi, qb_lo = _to16(q.contiguous(), precision, split)
        kv = torch.cat([kv_k, kv_v], dim=-1).contiguous()
        kv_hi, kv_lo = _to16(kv, precision, split)
        m.qk_hi = qb_hi.data_ptr()
        m.qk_lo = qb_lo.data_ptr() if split else None
        m.ld_qk, m.q_col0 = d, 0
        m.kv_hi = kv_hi.data_ptr()
        m.kv_lo = kv_lo.data_ptr() if split else None
        m.ld_kv, m.Tk, m.k_col0, m.v_col0 = 2 * d, Tk, 0, d
    else:
        assert Tk == T
        qk = torch.cat([q, kv_k, kv_v], dim=-1).contiguous()
        qk_hi, qk_lo = _to16(qk, precision, split)
        m.qk_hi = qk_hi.data_ptr()
        m.qk_lo = qk_lo.data_ptr() if split else None
        m.ld_qk, m.q_col0, m.k_col0, m.v_col0 = 3 * d, 0, d, 2 * d
    m.kv_len = kv_len.data_ptr()
    out_hi = torch.full((B, T, d), float('nan'), device=DEV, dtype=torch.bfloat16)
    out_lo = torch.full((B, T, d), float('nan'), device=DEV, dtype=torch.bfloat16)
    m.out_hi = out_hi.data_ptr()
    m.out_lo = out_lo.data_ptr()
    m.ld_out = d
    m.causal = int(causal)
    m.full_queries = int(full_queries)
    wts = None
    if weights_all:
        wts = torch.full((B, H, T, Tk), float('nan'), device=DEV)
        m.weights_out = wts.data_ptr()
        m.weights_all = 1
    m.precision = {'bf16x3': lib.PREC_BF16X3, 'bf16': lib.PREC_BF16, 'fp16': lib.PREC_FP16}[precision]
    m.impl = lib.IMPL_SIMT if impl == 'simt' else lib.IMPL_TCGEN05
    lib.mha_fwd(m)
    torch.cuda.synchronize()
    return out_hi.float() + out_lo.float(), wts


def ref_mha_general(q, k, v, kv_len, H, precision, causal=False):
    """float64 CPU attention; additive -1e9 mask = max(key padding, look-ahead) (models.py:136-138, layers.py:186-187)."""
    cast = {'bf16x3': lambda t: t.detach().cpu().double(), 'bf16': lambda t: t.detach().cpu().bfloat16().double(),
            'fp16': lambda t: t.detach().cpu().half().double()}[precision]
    q, k, v = cast(q), cast(k), cast(v)
    B, T, d = q.shape
    Tk = k.shape[1]
    dh = d // H
    sp = lambda t: t.reshape(B, t.shape[1], H, dh).permute(0, 2, 1, 3)
    logits = sp(q) @ sp(k).transpose(-1, -2) / (dh ** 0.5)
    mask = (torch.arange(Tk)[None, :] >= kv_len.cpu()[:, None]).double()[:, None, None, :].expand(B, 1, T, Tk)
    if causal:
        look = (torch.arange(Tk)[None, :] > torch.arange(T)[:, None]).double()[None, None]
        mask = torch.maximum(mask, look)
    logits = (logits.float() + (mask * -1e9).float()).double()
    w = torch.softmax(logits, -1)
    out = (w @ sp(v)).permute(0, 2, 1, 3).reshape(B, T, d)
    return out, w
