"""GPU parity of the training-step kernels one at a time.

Dropout is a stateless hash of (seed ^ salt, site, element index), drawn independently by every kernel that applies or
regenerates a mask.  Each site is checked against a host restatement of that hash (gpu_util.dropout_keep_host): the kept
set read off a forward output must EQUAL the host mask at the element index the site documents (include/ttsb.h), and every
backward kernel is compared with an fp64 reference built with the host mask.  The small backward kernels of the step
(expand / embedding / pitch embedding / statistics head, losses, ReLU mask, casts, Adam) and the batched weight repack are
checked against fp64 or exact host results at the model's shapes and their edges.

Gates: masks exact (plus a 5-sigma binomial check of the kept fraction, so a no-op mask cannot pass); integer and copy
results exact; fp32 results per element against fp64, with gates derived from the length of the sums; bf16 outputs within
one bf16 ulp of the fp64 value.  Every test prints its worst measured error next to its gate."""
import math

import numpy as np
import pytest
import torch

from gpu_util import DEV, dropout_keep_host, ref_gemm, run_gemm

pytestmark = pytest.mark.gpu

SALT = 0x2545F491          # a non-zero per-step salt (ttsb_set_dropout_salt)
U32 = 2.0 ** -24           # unit roundoff of fp32


def _lib():
    from transformertts_b200 import lib
    lib.load()
    return lib


def _set_salt(value):
    lib = _lib()
    salt = torch.tensor([value], dtype=torch.int32, device=DEV)
    lib.set_dropout_salt(salt)
    torch.cuda.synchronize()


@pytest.fixture(scope='module', autouse=True)
def _salt_back_to_zero():
    """Tests elsewhere in the process assume the library's salt is 0."""
    yield
    _set_salt(0)


def _gate(what, err, gate):
    print(f'{what}: worst {err:.3e}  (gate {gate:.1e})')
    assert err <= gate, (what, err, gate)


def _check_mask(kept, idx, p, seed, site, salt, what):
    """kept: bool array read off a kernel output; idx: the element indices of those entries."""
    want = dropout_keep_host(idx, p, seed, site, salt)
    kept = np.asarray(kept, dtype=bool)
    n = want.size
    mism = int((kept != want).sum())
    frac = float(kept.mean())
    five_sigma = 5 * math.sqrt(p * (1 - p) / n)
    print(f'{what}: {n} elements, {mism} mask mismatches, kept fraction {frac:.5f} (1-p = {1 - p}, 5 sigma {five_sigma:.1e})')
    assert mism == 0, (what, mism)
    assert abs(frac - (1 - p)) < five_sigma, (what, frac)


def _rel_to_max(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def _bf16_ulps(got, ref, floor):
    """worst |got - ref| in units of one bf16 ulp of the fp64 value ref; `floor` is the smallest ulp used (values that are
    fp32 rounding noise around zero)."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    ulp = torch.pow(2.0, torch.floor(torch.log2(ref.abs().clamp_min(1e-300))) - 7).clamp_min(floor)
    return float(((got - ref).abs() / ulp).max())


def _sum_bound(terms_abs_sum, n_terms):
    """a priori bound of fp32 summation: n * u * sum |terms| (any order, any atomics)"""
    return n_terms * U32 * terms_abs_sum


def _ln64(x, gamma, beta, eps=1e-6):
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * gamma + beta


def _inv_keep(p):
    return 1.0 / (1.0 - float(np.float32(p)))


# =====================================================================================================================
# B. forward sites: the kept set bit for bit
# =====================================================================================================================
@pytest.mark.parametrize('kind', ['embed', 'expand'])
@pytest.mark.parametrize('p,salt', [(0.1, 0), (0.25, 0), (0.1, SALT), (0.25, SALT)])
def test_prologue_dropout_mask_and_values(kind, p, salt):
    """embed_ln_pe / expand_ln_pe training forwards: element index = flat output index (b*T + t)*d + c."""
    lib = _lib()
    _set_salt(salt)
    g = torch.Generator().manual_seed(21)
    B, Tp, Tm, vocab = 3, 60, 250, 40
    d = 384 if kind == 'embed' else 256
    gamma, beta = 1 + 0.1 * torch.randn(d, generator=g), 0.5 + 0.1 * torch.rand(d, generator=g)
    pe, scalar = torch.randn(1000, d, generator=g), torch.tensor([0.7])
    seed, site = 987654321, 3
    if kind == 'embed':
        T = Tp
        emb = torch.randn(vocab, d, generator=g)
        tok = torch.randint(0, vocab, (B, T), generator=g, dtype=torch.int32)
        rows = emb.double()[tok.long()]
    else:
        T = Tm
        x = torch.randn(B, Tp, d, generator=g)
        dur = torch.randint(1, 6, (B, Tp), generator=g)
        idx = torch.full((B, Tm), -1, dtype=torch.int32)
        for b in range(B):
            rep = torch.repeat_interleave(torch.arange(Tp), dur[b])[:Tm - 7 * b]       # padded tail frames (-1) in rows 1, 2
            idx[b, :len(rep)] = rep.int()
        rows = torch.where((idx >= 0)[..., None], x.double()[torch.arange(B)[:, None], idx.clamp_min(0).long()],
                           torch.zeros((), dtype=torch.float64))
    ref = _ln64(rows, gamma.double(), beta.double()) + 0.7 * pe.double()[:T]
    out = torch.full((B, T, d), float('nan'), device=DEV)
    hi = torch.full((B, T, d), float('nan'), dtype=torch.bfloat16, device=DEV)
    args = (gamma.to(DEV), beta.to(DEV), pe.to(DEV), scalar.to(DEV), 1e-6, out, hi, None)
    if kind == 'embed':
        lib.embed_ln_pe_fwd(tok.to(DEV), emb.to(DEV), *args, drop=(p, seed, site))
    else:
        lib.expand_ln_pe_fwd(x.to(DEV), idx.to(DEV), *args, drop=(p, seed, site))
    torch.cuda.synchronize()
    assert (ref != 0).all()                                                   # a zero output element is a dropped one
    o = out.cpu()
    flat = np.arange(B * T * d, dtype=np.uint64).reshape(B, T, d)
    _check_mask((o != 0).numpy(), flat, p, seed, site, salt, f'{kind}_ln_pe site')
    assert torch.equal(hi.cpu() != 0, o != 0)
    want = ref * (o != 0) * _inv_keep(p)
    _gate(f'{kind}_ln_pe fp32 vs fp64 (rel. to max)', _rel_to_max(o, want), 2e-6)
    _gate(f'{kind}_ln_pe bf16 hi (bf16 ulps)', _bf16_ulps(hi.float(), want, 1e-5 * float(want.abs().max())), 1.0)


@pytest.mark.parametrize('N,staged', [(256, False), (256, True), (226, False)])
@pytest.mark.parametrize('p,salt', [(0.1, 0), (0.25, SALT)])
def test_linear_fwd_drop_pre_mask(N, staged, p, salt):
    """Dense GEMM with drop_pre (no residual, no ReLU, so every kept output is non-zero): element index
    (b*T + t)*ld_out + n, through the direct epilogue (fp32 output) and the staged 16-bit tile-store epilogue."""
    _set_salt(salt)
    g = torch.Generator().manual_seed(22)
    B, T, K = 3, 300, 256
    x = torch.randn(B, T, K, generator=g).to(DEV)
    w = (torch.randn(K, N, generator=g) / 16).to(DEV)
    bias = (0.1 * torch.randn(N, generator=g)).to(DEV)
    seed, site = 4242, 9
    o = run_gemm([x], w, bias, [0], [0], [K], precision='bf16', drop_pre=(p, site), drop_seed=seed, want_f32=not staged)
    ld = o['n_pad']
    ref = ref_gemm([x], w, bias, [0], [0], [K], precision='bf16', drop_pre=(p, site), drop_seed=seed, salt=salt, ld_out=ld)
    got = (o['hi'] if staged else o['f32']).float().cpu()
    assert (got[..., N:] == 0).all()
    got = got[..., :N]
    idx = (np.arange(B * T, dtype=np.uint64)[:, None] * np.uint64(ld) + np.arange(N, dtype=np.uint64)[None, :]).reshape(B, T, N)
    _check_mask((got != 0).numpy(), idx, p, seed, site, salt, f'linear_fwd drop_pre ({"staged" if staged else "direct"})')
    floor = 1e-5 * float(ref.abs().max())
    if staged:
        _gate('linear_fwd drop_pre bf16 (bf16 ulps)', _bf16_ulps(got, ref, floor), 1.0)
    else:
        _gate('linear_fwd drop_pre fp32 vs fp64 (rel. to max)', _rel_to_max(got, ref), 3e-6)
        _gate('linear_fwd drop_pre bf16 hi (bf16 ulps)', _bf16_ulps(o['hi'].float().cpu()[..., :N], ref, floor), 1.0)


# row tiles of 128 rows: <= 74 -> CTA pairs; 148 -> single-CTA tiles; 200 -> 148 single-CTA tiles + a pair tail (148 SMs)
_SCHEDULES = {'pair': (4, 300), 'single': (74, 256), 'hybrid': (100, 256)}


@pytest.mark.parametrize('schedule', ['pair', 'single', 'hybrid'])
@pytest.mark.parametrize('p', [0.0, 0.1])
def test_linear_fwd_residual_layernorm_schedules(schedule, p):
    """Residual + LayerNorm GEMM at N = d = 256 with both dropout sites, on every schedule of the LayerNorm epilogue:
    out_f32 / out_hi / out_preln against fp64 with the host masks, and the kept set of drop_post exactly."""
    lib = _lib()
    _set_salt(0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != 148:
        pytest.skip(f'row-tile counts are chosen for 148 SMs (this device has {sms})')
    g = torch.Generator().manual_seed(23)
    B, T = _SCHEDULES[schedule]
    K = N = 256
    x = torch.randn(B, T, K, generator=g).to(DEV)
    w = (torch.randn(K, N, generator=g) / 16).to(DEV)
    bias = (0.1 * torch.randn(N, generator=g)).to(DEV)
    res = torch.randn(B, T, N, generator=g).to(DEV)
    gam, bet = (1 + 0.1 * torch.randn(N, generator=g)).to(DEV), (0.1 * torch.randn(N, generator=g)).to(DEV)
    seed, pre, post = 777, 5, 6
    o = run_gemm([x], w, bias, [0], [0], [K], precision='bf16', residual=res, ln=(gam, bet), drop_pre=(p, pre),
                 drop_post=(p, post), drop_seed=seed, out_preln=True, single_tile=True)
    assert o['launches'] == (2 if schedule == 'hybrid' else 1), o['launches']
    ref, ref_pre = ref_gemm([x], w, bias, [0], [0], [K], precision='bf16', residual=res, ln=(gam, bet), drop_pre=(p, pre),
                            drop_post=(p, post), drop_seed=seed, ld_out=o['n_pad'], return_preln=True)
    f32, preln = o['f32'].cpu(), o['preln'].cpu()
    _gate(f'{schedule} p={p} out_preln vs fp64 (rel. to max)', _rel_to_max(preln, ref_pre), 3e-6)
    _gate(f'{schedule} p={p} out_f32 vs fp64 (rel. to max)', _rel_to_max(f32, ref), 1e-5)
    _gate(f'{schedule} p={p} out_hi (bf16 ulps)', _bf16_ulps(o['hi'].float(), ref, 2e-5 * float(ref.abs().max())), 1.0)
    if p > 0:
        idx = np.arange(B * T * N, dtype=np.uint64).reshape(B, T, N)
        _check_mask((f32 != 0).numpy(), idx, p, seed, post, 0, f'{schedule} drop_post')


def _softmax64(S, B, H, T, lens):
    """fp64 softmax of rows (Z,T,ld) over keys < len; query rows t >= len are zero"""
    Z, _, ld = S.shape
    k = torch.arange(ld)[None, None, :]
    klen = lens.repeat_interleave(H)[:, None, None]
    valid = (k < klen) & (torch.arange(T)[None, :, None] < klen)
    s = S.double().masked_fill(~valid, float('-inf'))
    P = torch.softmax(s, -1).nan_to_num(0.0)
    return P * valid, valid


@pytest.mark.parametrize('T,p,salt', [(333, 0.25, 0), (1000, 0.1, SALT), (1100, 0.1, 0), (1200, 0.25, SALT), (1300, 0.1, 0)])
def test_softmax_fwd_and_attn_probs_dropout_mask(T, p, salt):
    """ttsb_softmax_fwd (vector kernel for ld <= 1024, scalar kernel above: the shipped config trains buckets up to 1200
    frames and beyond) and ttsb_attn_probs_fwd: element index (z*T + t)*ld + key."""
    lib = _lib()
    _set_salt(salt)
    from transformertts_b200.model.models import _round_up
    g = torch.Generator().manual_seed(24)
    B, H, dh = 2, 2, 128
    Z, ld = B * H, _round_up(T, 16)
    lens = torch.tensor([T, T // 2 + 7], dtype=torch.int32)
    S = 2 * torch.randn(Z, T, ld, generator=g)
    seed, site = 31337, 12
    Pp = torch.full((Z, T, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    Pd = torch.full((Z, T, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    lib.softmax_fwd(S.to(DEV), B, H, T, T, ld, lens.to(DEV), p, seed, site, Pp, Pd)
    torch.cuda.synchronize()
    ref, valid = _softmax64(S, B, H, T, lens)
    pp, pd = Pp.float().cpu(), Pd.float().cpu()
    floor = 2.0 ** -40
    _gate(f'softmax_fwd T={T} P_pre (bf16 ulps)', _bf16_ulps(pp, ref, floor), 1.0)
    assert (pd[~valid] == 0).all()
    idx = np.arange(Z * T * ld, dtype=np.uint64).reshape(Z, T, ld)
    _check_mask((pd != 0).numpy()[valid.numpy()], idx[valid.numpy()], p, seed, site, salt, f'softmax_fwd T={T}')
    want = ref * (pd != 0) * _inv_keep(p)
    _gate(f'softmax_fwd T={T} P_drop (bf16 ulps)', _bf16_ulps(pd, want, floor), 1.0)
    # the fused kernel on Q K^T of bf16 activations
    d = H * dh
    qkv = torch.randn(B, T, 3 * d, generator=g).bfloat16()
    if not lib.attn_probs_supported(dh, ld):
        with pytest.raises(lib.TtsbError):
            lib.attn_probs_fwd(qkv.to(DEV), 3 * d, 0, d, B, H, T, dh, lens.to(DEV), 1.0 / math.sqrt(dh), p, seed, site, Pp, Pd, ld)
        return
    Pp.fill_(float('nan'))
    Pd.fill_(float('nan'))
    lib.attn_probs_fwd(qkv.to(DEV), 3 * d, 0, d, B, H, T, dh, lens.to(DEV), 1.0 / math.sqrt(dh), p, seed, site, Pp, Pd, ld)
    torch.cuda.synchronize()
    q, k = [t.reshape(B, T, H, dh).permute(0, 2, 1, 3).reshape(Z, T, dh) for t in qkv.double().split(d, dim=-1)[:2]]
    S2 = torch.zeros(Z, T, ld, dtype=torch.float64)
    S2[..., :T] = q @ k.transpose(-1, -2) / math.sqrt(dh)
    ref2, _ = _softmax64(S2, B, H, T, lens)
    pp, pd = Pp.float().cpu(), Pd.float().cpu()
    assert (pd[~valid] == 0).all() and (pp[~valid] == 0).all()
    live = valid & (pp != 0)
    _check_mask((pd != 0).numpy()[live.numpy()], idx[live.numpy()], p, seed, site, salt, f'attn_probs_fwd T={T}')
    want2 = ref2 * (pd != 0) * _inv_keep(p)
    err = float(((pd.double() - want2).abs() / (want2 + 1e-6))[live].max())
    _gate(f'attn_probs_fwd T={T} P_drop relative', err, 6e-3)       # bf16 rounding (2^-9) + ex2.approx, as the P_pre test


# =====================================================================================================================
# C. backward sites: fp64 with the host mask
# =====================================================================================================================
@pytest.mark.parametrize('kernel', ['vector', 'scalar'])
@pytest.mark.parametrize('site_kind,p,salt', [('post', 0.1, 0), ('pre', 0.1, 0), ('post', 0.25, SALT), ('pre', 0.25, SALT)])
def test_layernorm_bwd_dropout(kernel, site_kind, p, salt):
    """ttsb_layernorm_bwd with post_drop (mask on dz) or pre_drop (mask on g_bf16): du, g_bf16, dgamma, dbeta, dbias
    against fp64 with the host mask; vector kernel C = ld = 256, scalar kernel C = 226, ld = 256 with the ReLU mask."""
    lib = _lib()
    _set_salt(salt)
    g = torch.Generator().manual_seed(25)
    B, T, ld = 4, 333, 256
    C = 256 if kernel == 'vector' else 226
    relu = kernel == 'scalar'
    u = torch.zeros(B, T, ld)
    dz = torch.zeros(B, T, ld)
    u[..., :C] = torch.randn(B, T, C, generator=g)
    dz[..., :C] = torch.randn(B, T, C, generator=g)
    gamma = torch.zeros(ld)
    gamma[:C] = 1 + 0.1 * torch.randn(C, generator=g)
    lens = torch.tensor([333, 100, 0, 250], dtype=torch.int32)
    seed, site = 55555, 17
    idx = np.arange(B * T * ld, dtype=np.uint64).reshape(B, T, ld)
    keep = torch.from_numpy(dropout_keep_host(idx, p, seed, site, salt)).double() * _inv_keep(p)
    live = (torch.arange(T)[None] < lens[:, None])[..., None].double()
    gz = dz.double()[..., :C] * live * (keep[..., :C] if site_kind == 'post' else 1.0)
    uu = u.double()[..., :C]
    mean = uu.mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(((uu - mean) ** 2).mean(-1, keepdim=True) + 1e-6)
    xh = (uu - mean) * rstd
    gg = gz * gamma.double()[:C]
    du_ref = rstd * (gg - gg.mean(-1, keepdim=True) - xh * (gg * xh).mean(-1, keepdim=True))
    gv = du_ref * ((uu > 0).double() if relu else 1.0) * (keep[..., :C] if site_kind == 'pre' else 1.0)
    du = torch.full((B, T, ld), float('nan'), device=DEV)
    gb = torch.full((B, T, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    dg, db, dbias = torch.zeros(ld, device=DEV), torch.zeros(ld, device=DEV), torch.zeros(ld, device=DEV)
    drop = dict(post_drop=(p, site)) if site_kind == 'post' else dict(pre_drop=(p, site))
    lib.layernorm_bwd(dz.to(DEV), u.to(DEV), gamma.to(DEV), B, T, C, ld, 1e-6, lens.to(DEV), relu, du, gb, dg, db, seed=seed,
                      dbias=dbias, **drop)
    torch.cuda.synchronize()
    du, gb = du.cpu(), gb.float().cpu()
    assert (du[..., C:] == 0).all() and (gb[..., C:] == 0).all()
    tag = f'layernorm_bwd {kernel} {site_kind} p={p}'
    _gate(f'{tag} du (rel. to max)', _rel_to_max(du[..., :C], du_ref), 2e-6)
    _gate(f'{tag} g_bf16 (bf16 ulps)', _bf16_ulps(gb[..., :C], gv, 1e-5 * float(gv.abs().max())), 1.0)
    rows = B * T
    for name, got, ref in (('dgamma', dg, (gz * xh).sum((0, 1))), ('dbeta', db, gz.sum((0, 1))), ('dbias', dbias, gv.sum((0, 1)))):
        terms = {'dgamma': (gz * xh).abs(), 'dbeta': gz.abs(), 'dbias': gv.abs()}[name].sum((0, 1))
        err = float(((got.cpu()[:C].double() - ref).abs() / _sum_bound(terms, rows).clamp_min(1e-30)).max())
        _gate(f'{tag} {name} (fraction of the fp32 summation bound)', err, 1.0)
    if site_kind == 'pre':   # the kept set of g_bf16 on live rows (where du != 0 and, with the ReLU mask, u > 0)
        sel = ((live[..., 0] > 0)[..., None] & (du_ref != 0) & ((uu > 0) if relu else True)).numpy()
        _check_mask((gb[..., :C] != 0).numpy()[sel], idx[..., :C][sel], p, seed, site, salt, tag)


@pytest.mark.parametrize('d', [128, 256, 384, 130, 1544])
def test_pe_scalar_bwd_dropout(d):
    """d(pos_encoding_scalar) = sum dropout(g) * PE[t] at C3 size (32 x 1000 rows; 4 x 1000 for the widest row): the vector
    kernel (d % 4 == 0, d/4 <= 384) and the scalar kernel (d = 130, d = 1544), against fp64 with the host mask."""
    lib = _lib()
    _set_salt(0)
    g = torch.Generator().manual_seed(26)
    B, T = (4, 1000) if d > 1536 else (32, 1000)
    gr = torch.randn(B, T, d, generator=g)
    pe = torch.randn(T, d, generator=g)
    p, seed, site = 0.1, 2024, 2
    keep = torch.from_numpy(dropout_keep_host(np.arange(B * T * d, dtype=np.uint64), p, seed, site)).view(B, T, d)
    terms = gr.double() * keep * _inv_keep(p) * pe.double()[None]
    ref = float(terms.sum())
    out = torch.zeros(1, device=DEV)
    lib.pe_scalar_bwd(gr.to(DEV), pe.to(DEV), out, drop=(p, seed, site))
    torch.cuda.synchronize()
    # the result is one fp32 sum of B*T*d products, accumulated per thread, then by warp / block trees and atomics: its
    # error is ~1e-9 of sum |terms|, gate 1e-7 (a mask error in a quarter of the elements moves the sum by ~5e-4 of it)
    err = abs(out.item() - ref) / float(terms.abs().sum())
    _gate(f'pe_scalar_bwd d={d} (fraction of sum |terms|)', err, 1e-7)


def _attn_bwd_inputs(T, dh, g):
    from transformertts_b200.model.models import _round_up
    B, H = 2, 2
    d, Z, ld = H * dh, B * H, _round_up(T, 16)
    lens = torch.tensor([T, T // 2 + 5], dtype=torch.int32)
    qkv = torch.randn(B, T, 3 * d, generator=g).bfloat16()
    dO = torch.randn(B, T, d, generator=g).bfloat16()
    kmask = (torch.arange(ld)[None, :] < lens[:, None]).repeat_interleave(H, 0)[:, None, :]
    qmask = (torch.arange(T)[None, :] < lens[:, None]).repeat_interleave(H, 0)[:, :, None]
    P = torch.rand(Z, T, ld, generator=g)
    P = (P * kmask * qmask / P.sum(-1, keepdim=True).clamp_min(1e-3)).bfloat16()
    D = torch.randn(Z * T, generator=g) * 0.1
    v = qkv.double()[..., 2 * d:].reshape(B, T, H, dh).permute(0, 2, 1, 3).reshape(Z, T, dh)
    do = dO.double().reshape(B, T, H, dh).permute(0, 2, 1, 3).reshape(Z, T, dh)
    dP = torch.zeros(Z, T, ld, dtype=torch.float64)
    dP[:, :, :T] = do @ v.transpose(-1, -2)
    return B, H, d, Z, ld, lens, qkv, dO, P, D, dP, (kmask & qmask)


@pytest.mark.parametrize('T,dh,salt', [(333, 64, 0), (1000, 128, SALT), (1200, 128, 0)])
def test_softmax_bwd_sites_against_fp64(T, dh, salt):
    """ttsb_softmax_bwd, the hashed dS epilogue of ttsb_bgemm (sm_Pdrop = NULL) and ttsb_attn_ds_bwd, each against
    dS = scale * P * (keep * dP / (1-p) - D) in fp64 with the host mask at element index (z*T + t)*ld + key."""
    lib = _lib()
    _set_salt(salt)
    from transformertts_b200.model.training import TrainEngine
    g = torch.Generator().manual_seed(27)
    B, H, d, Z, ld, lens, qkv, dO, P, D, dP, live = _attn_bwd_inputs(T, dh, g)
    p, seed, site, scale = 0.1, 8080, 4, 1.0 / math.sqrt(dh)
    keep = torch.from_numpy(dropout_keep_host(np.arange(Z * T * ld, dtype=np.uint64), p, seed, site, salt)).view(Z, T, ld)
    gk = keep * dP * _inv_keep(p)
    # softmax_bwd computes its own row statistic D = sum_k P * keep * dP / (1-p) from the fp32 dP
    dS_ref = scale * P.double() * (gk - (P.double() * gk * live).sum(-1, keepdim=True)) * live
    lens_d, P_d = lens.to(DEV), P.to(DEV)
    dS = torch.full((Z, T, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    lib.softmax_bwd(P_d, dP.float().to(DEV), B, H, T, T, ld, lens_d, scale, p, seed, site, dS)
    torch.cuda.synchronize()
    # dP is rounded to fp32 first: its rounding (u * |dP|) and the fp32 row sum set the floor of the ulp comparison
    floor = 1e-5 * float(dS_ref.abs().max())
    _gate(f'softmax_bwd T={T} (bf16 ulps)', _bf16_ulps(dS.float(), dS_ref, floor), 1.0)
    # the fused forms take D = dO . O from outside
    ref = scale * P.double() * (gk - D.double().view(Z, T, 1)) * live
    floor = 1e-5 * float(ref.abs().max())
    eng = TrainEngine.__new__(TrainEngine)
    eng.dev = torch.device(DEV)
    qkv_d, dO_d, D_d = qkv.to(DEV), dO.to(DEV), D.to(DEV)
    dS0 = torch.full((Z, T, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    eng._bgemm(B, H, T, T, dh, dO_d, (d, T, B), (d, d * T), (dh, 0, 0, 0), qkv_d, (d, T, B), (3 * d, 3 * d * T), (dh, 0, 0, 2 * d),
               out_bf16=dS0, ld_out=ld, out_batch_stride=T * ld, out_cols=ld,
               softmax_bwd=(P_d, D_d, scale, p, seed, site, 0, lens_d, None))
    torch.cuda.synchronize()
    _gate(f'bgemm dS epilogue T={T} (bf16 ulps)', _bf16_ulps(dS0.float(), ref, floor), 1.0)
    dS1 = torch.full((Z, T, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    assert lib.attn_probs_supported(dh, ld)
    lib.attn_ds_bwd(dO_d, d, 0, qkv_d, 3 * d, 2 * d, B, H, T, dh, lens_d, P_d, D_d, scale, p, seed, site, dS1, ld)
    torch.cuda.synchronize()
    _gate(f'attn_ds_bwd T={T} (bf16 ulps)', _bf16_ulps(dS1.float(), ref, floor), 1.0)


# =====================================================================================================================
# D. the other backward kernels at the model's shapes and their edges
# =====================================================================================================================
@pytest.mark.parametrize('Tp,d', [(57, 384), (300, 256), (1500, 128)])
def test_expand_bwd(Tp, d):
    """dx[b,i] = sum of dm[b,t] over the frames of phoneme i: multi-pass block scan (Tp > 256), several row chunks, zero and
    negative durations, rows truncated at Tm, odd segment lengths; gate = fp32 rounding of the (short) sums."""
    lib = _lib()
    g = torch.Generator().manual_seed(28)
    B = 3
    dur = torch.randint(-2, 8, (B, Tp), generator=g, dtype=torch.int32)
    tot = dur.clamp_min(0).sum(1)
    Tm = int(tot[0]) + 3                                   # row 0 fits with padding frames; rows 1, 2 may be truncated
    dur[1] = dur[1].abs() + 1                              # row 1: sum(dur) > Tm (truncated)
    if int(dur[1].sum()) <= Tm:
        dur[1, -1] += Tm - int(dur[1].sum()) + 10
    dm = torch.randn(B, Tm, d, generator=g)
    start = torch.cumsum(dur.clamp_min(0), 1) - dur.clamp_min(0)
    ref = torch.zeros(B, Tp, d, dtype=torch.float64)
    bound = torch.zeros(B, Tp, d, dtype=torch.float64)
    dm64 = dm.double()
    for b in range(B):
        for i in range(Tp):
            s, e = min(int(start[b, i]), Tm), min(int(start[b, i] + dur[b, i].clamp_min(0)), Tm)
            if e > s:
                ref[b, i] = dm64[b, s:e].sum(0)
                bound[b, i] = (e - s) * U32 * dm64[b, s:e].abs().sum(0)
    assert int(dur[1].clamp_min(0).sum()) > Tm and (dur == 0).any() and (dur < 0).any() and (dur % 2 == 1).any()
    dx = torch.full((B, Tp, d), float('nan'), device=DEV)
    lib.expand_bwd(dm.to(DEV), dur.to(DEV), dx)
    torch.cuda.synchronize()
    dx = dx.cpu().double()
    assert torch.isfinite(dx).all()
    assert (dx[ref == 0] == 0).all()                       # empty segments (zero / negative / truncated) are written as 0
    err = float(((dx - ref).abs() - bound).max())
    print(f'expand_bwd Tp={Tp} d={d}: worst error beyond the summation bound {err:.3e} (gate 0)')
    assert err <= 0.0


def test_embedding_bwd_repeated_and_clamped_tokens():
    """demb[tok] += dx rows: heavily repeated tokens (atomics), ids 0 and vocab-1, and out-of-range ids clamped."""
    lib = _lib()
    g = torch.Generator().manual_seed(29)
    B, T, d, vocab = 4, 300, 256, 50
    tok = torch.randint(0, vocab, (B, T), generator=g, dtype=torch.int32)
    tok[:, ::3] = 0
    tok[:, 1::7] = vocab - 1
    tok[0, :5] = torch.tensor([-1, -7, vocab, vocab + 3, 2 ** 30], dtype=torch.int32)
    dx = torch.randn(B, T, d, generator=g)
    ids = tok.clamp(0, vocab - 1).long().view(-1)
    ref = torch.zeros(vocab, d, dtype=torch.float64).index_add_(0, ids, dx.double().view(-1, d))
    cnt = torch.bincount(ids, minlength=vocab).double()[:, None]
    bound = cnt * U32 * torch.zeros(vocab, d, dtype=torch.float64).index_add_(0, ids, dx.double().abs().view(-1, d))
    demb = torch.zeros(vocab, d, device=DEV)
    lib.embedding_bwd(dx.to(DEV), tok.to(DEV), demb)
    torch.cuda.synchronize()
    err = float(((demb.cpu().double() - ref).abs() / bound.clamp_min(1e-30)).max())
    _gate('embedding_bwd (fraction of the fp32 summation bound)', err, 1.0)
    assert int(cnt[0]) > 300 and int(cnt[vocab - 1]) > 150


@pytest.mark.parametrize('d', [384, 600])
def test_pitch_embed_bwd(d):
    """dw / db of Dense(1 -> d, relu): 231 rows (not a multiple of 64), d = 384 and d = 600 (> 512: strided channel loop),
    pre-activations exactly 0 carry no gradient (TF's ReLU)."""
    lib = _lib()
    g = torch.Generator().manual_seed(30)
    B, T = 3, 77
    gr = torch.randn(B, T, d, generator=g)
    pitch = torch.randn(B, T, generator=g)
    w, bias = torch.randn(d, generator=g), 0.5 * torch.randn(d, generator=g)
    pitch[0, :4] = 0.0
    bias[:8] = 0.0                                         # pitch 0, bias 0: pre-activation exactly 0
    pitch[1, :4] = 1.0
    bias[8:16] = -w[8:16]                                  # pitch 1: w + b exactly 0
    pre = pitch.double()[..., None] * w.double() + bias.double()
    m = (pre > 0).double()
    assert ((pre == 0).sum()) >= 64
    g64 = gr.double()
    rows = B * T
    dw_ref = (g64 * m * pitch.double()[..., None]).sum((0, 1))
    db_ref = (g64 * m).sum((0, 1))
    dw, db = torch.zeros(d, device=DEV), torch.zeros(d, device=DEV)
    lib.pitch_embed_bwd(gr.to(DEV), pitch.to(DEV), w.to(DEV), bias.to(DEV), dw, db)
    torch.cuda.synchronize()
    for name, got, ref, terms in (('dw', dw, dw_ref, (g64 * m * pitch.double()[..., None]).abs().sum((0, 1))),
                                  ('db', db, db_ref, (g64 * m).abs().sum((0, 1)))):
        err = float(((got.cpu().double() - ref).abs() / _sum_bound(terms, rows).clamp_min(1e-30)).max())
        _gate(f'pitch_embed_bwd d={d} {name} (fraction of the fp32 summation bound)', err, 1.0)


@pytest.mark.parametrize('relu', [True, False])
def test_statpred_head_bwd(relu):
    """StatPredictor head Dense(C -> 1) * mask backward: ReLU on / off, row_len 0 / partial / full, ldh > C with dh zero in
    columns C..ldh; dh is one product per element (exact), dw / db fp32 sums."""
    lib = _lib()
    g = torch.Generator().manual_seed(31)
    B, T, C, ldh = 3, 90, 226, 256
    gout = torch.randn(B, T, generator=g)
    out = torch.randn(B, T, generator=g)
    out[0, :6] = 0.0                                       # relu'(0) = 0
    h = torch.randn(B, T, ldh, generator=g)
    w = torch.randn(C, generator=g)
    lens = torch.tensor([0, 37, T], dtype=torch.int32)
    gm = gout * (torch.arange(T)[None] < lens[:, None]) * ((out > 0) if relu else 1.0)
    dh_ref = torch.zeros(B, T, ldh)
    dh_ref[..., :C] = (gm.double()[..., None] * w.double()).float()
    dw_ref = (gm.double()[..., None] * h.double()[..., :C]).sum((0, 1))
    db_ref = gm.double().sum()
    dh = torch.full((B, T, ldh), float('nan'), device=DEV)
    dw, db = torch.zeros(C, device=DEV), torch.zeros(1, device=DEV)
    lib.statpred_head_bwd(gout.to(DEV), out.to(DEV), h.to(DEV), C, w.to(DEV), relu, lens.to(DEV), dh, dw, db)
    torch.cuda.synchronize()
    assert torch.equal(dh.cpu(), dh_ref)
    rows = B * T
    err = float(((dw.cpu().double() - dw_ref).abs() / _sum_bound((gm.double()[..., None] * h.double()[..., :C]).abs().sum((0, 1)),
                                                                  rows)).max())
    _gate(f'statpred_head_bwd relu={relu} dw (fraction of the fp32 summation bound)', err, 1.0)
    err = abs(db.item() - float(db_ref)) / _sum_bound(float(gm.double().abs().sum()), rows)
    _gate(f'statpred_head_bwd relu={relu} db (fraction of the fp32 summation bound)', err, 1.0)


def test_mae_loss_float_targets_shorter_than_prediction():
    """The mel loss: float targets, Tt < Tp (rows t >= Tt carry no loss and zero gradient), pred == target gives a zero
    gradient; the gradient is exact, the loss an fp32 sum."""
    lib = _lib()
    g = torch.Generator().manual_seed(32)
    B, Tp, Tt, C = 3, 210, 170, 80
    pred = torch.randn(B, Tp, C, generator=g)
    tgt = torch.randn(B, Tt, C, generator=g)
    tgt[:, :9] = pred[:, :9, :]
    n = B * Tt * C
    weight = 1.0
    diff = pred[:, :Tt].double() - tgt.double()
    loss_ref = float(diff.abs().sum() / n)
    grad_ref = torch.zeros(B, Tp, C)
    grad_ref[:, :Tt] = torch.sign(diff).float() * np.float32(weight) * (np.float32(1.0) / np.float32(n))
    loss = torch.zeros(1, device=DEV)
    grad = torch.full((B, Tp, C), float('nan'), device=DEV)
    lib.mae_loss(pred.to(DEV), B, Tp, Tt, C, tgt.to(DEV), weight, loss, grad)
    torch.cuda.synchronize()
    assert torch.equal(grad.cpu(), grad_ref)
    assert (grad.cpu()[:, :9] == 0).all()
    _gate('mae_loss (relative)', abs(loss.item() - loss_ref) / loss_ref, 1e-6)


def test_diag_loss_train():
    """Training form of the Aligner's diagonal loss on bf16 P with ld > Tk and a zero key length: the loss and the dP
    increment against fp64 (the increment is one fp32 multiply-add per element)."""
    lib = _lib()
    g = torch.Generator().manual_seed(33)
    B, H, Tq, Tk, ld = 3, 2, 70, 45, 64
    P = torch.rand(B * H, Tq, ld, generator=g).bfloat16()
    q_len = torch.tensor([70, 33, 50], dtype=torch.int32)
    k_len = torch.tensor([45, 20, 0], dtype=torch.int32)
    dP0 = torch.randn(B * H, Tq, ld, generator=g)
    ls, gs = 1.5, 0.75
    inv = np.float32(1.0) / (np.float32(10.0) * np.float32(B * H))
    m = torch.zeros(B * H, Tq, ld, dtype=torch.float64)
    for z in range(B * H):
        b = z // H
        qm, kn = int(q_len[b]), int(k_len[b])
        if qm > 0 and kn > 0:
            qq = torch.arange(qm, dtype=torch.float64)[:, None] / qm
            kk = torch.arange(kn, dtype=torch.float64)[None, :] / kn
            m[z, :qm, :kn] = (kk - qq).abs().float().double()
    loss_ref = float(np.float32(ls) * inv) * float((P.double() * m).sum())
    dP_ref = dP0.double() + float(np.float32(gs) * inv) * m
    loss = torch.zeros(1, device=DEV)
    dP = dP0.to(DEV)
    lib.diag_loss_train(P.to(DEV), B, H, Tq, Tk, ld, q_len.to(DEV), k_len.to(DEV), ls, loss, gs, dP)
    torch.cuda.synchronize()
    dP = dP.cpu()
    assert torch.equal(dP[m == 0], dP0[m == 0])
    incr = dP_ref - dP0.double()
    err = float(((dP.double() - dP_ref).abs() / (dP0.double().abs() + incr.abs()))[m != 0].max())
    _gate('diag_loss_train dP (units of u * (|dP| + |increment|))', err / U32, 2.0)   # a product and a sum, or one fma
    _gate('diag_loss_train loss (relative)', abs(loss.item() - loss_ref) / loss_ref, 1e-6)


def test_relu_bwd_cast_and_rowdot():
    """relu_bwd: exact mask with h = +0 and -0 masked; cast_bf16_pad 80 -> 128 columns (exact, zero padding);
    rowdot_heads against fp64."""
    lib = _lib()
    g = torch.Generator().manual_seed(34)
    dy = torch.randn(64, 256, generator=g).bfloat16()
    h = torch.randn(64, 256, generator=g).bfloat16()
    h[:, :8] = 0.0
    h[:, 8:16] = -0.0
    assert (torch.signbit(h[:, 8:16].float())).all()
    dy_d = dy.to(DEV)
    lib.relu_bwd(dy_d, h.to(DEV))
    torch.cuda.synchronize()
    want = torch.where(h.float() > 0, dy.float(), torch.zeros(()))
    assert torch.equal(dy_d.float().cpu(), want) and (dy_d.cpu()[:, :16] == 0).all()
    x = torch.randn(3 * 77, 80, generator=g)
    out = torch.full((3 * 77, 128), float('nan'), dtype=torch.bfloat16, device=DEV)
    lib.cast_bf16_pad(x.to(DEV), 3 * 77, 80, out, 128)
    torch.cuda.synchronize()
    want = torch.zeros(3 * 77, 128, dtype=torch.bfloat16)
    want[:, :80] = x.bfloat16()
    assert torch.equal(out.cpu().view(torch.int16), want.view(torch.int16))
    B, T, H, dh = 2, 77, 4, 64
    xa = torch.randn(B, T, H * dh, generator=g).bfloat16()
    ya = torch.randn(B, T, H * dh, generator=g).bfloat16()
    D = torch.full((B * H * T,), float('nan'), device=DEV)
    lib.rowdot_heads(xa.to(DEV), ya.to(DEV), H, dh, D)
    torch.cuda.synchronize()
    prod = (xa.double() * ya.double()).view(B, T, H, dh)
    ref = prod.sum(-1).permute(0, 2, 1).reshape(-1)
    bound = _sum_bound(prod.abs().sum(-1).permute(0, 2, 1).reshape(-1), dh)
    _gate('rowdot_heads (fraction of the fp32 summation bound)', float(((D.cpu().double() - ref).abs() / bound).max()), 1.0)


def test_adam_grad_scale():
    """ttsb_adam_tf_step with grad_scale = 1/2 (data parallelism folds the 1/N of the gradient mean in here): moments and
    parameters against the Keras formula in fp64 on the same fp32 inputs, three steps."""
    lib = _lib()
    g = torch.Generator().manual_seed(35)
    n = 10000
    p0 = torch.randn(n, generator=g)
    grads = [torch.randn(n, generator=g) * 1e-2 for _ in range(3)]
    lr, b1, b2, eps, gs = 1e-3, 0.9, 0.98, 1e-9, 0.5
    pd, md, vd = p0.to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    pr, mr, vr = p0.double(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    f32 = lambda v: float(np.float32(v))                     # the kernel's scalars are fp32 (1 - 0.98f is 0.02 - 1.9e-8)
    b1f, b2f, c1f, c2f = f32(b1), f32(b2), f32(np.float32(1) - np.float32(b1)), f32(np.float32(1) - np.float32(b2))
    for t, gr in enumerate(grads, 1):
        lr_t = lr * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)
        lib.adam_tf_step(pd, gr.to(DEV), md, vd, lr_t, b1, b2, eps, grad_scale=gs)
        gg = gr.double() * gs
        mr = b1f * mr + c1f * gg
        vr = b2f * vr + c2f * gg * gg
        pr = pr - f32(lr_t) * mr / (vr.sqrt() + f32(eps))
    torch.cuda.synchronize()
    # a wrong grad_scale moves m by half of itself and v by three quarters; fp32 rounding of three steps is ~1e-7
    _gate('adam m (rel. to max)', _rel_to_max(md, mr), 1e-6)
    _gate('adam v (rel. to max)', _rel_to_max(vd, vr), 1e-6)
    # parameters: fp32 storage of p (|p| ~ 1) after three updates of ~lr each: a few fp32 ulps of |p| + lr
    err = float(((pd.cpu().double() - pr).abs() / ((pr.abs() + lr) * 2 ** -23)).max())
    _gate('adam param (fp32 ulps of |p| + lr)', err, 4.0)


# =====================================================================================================================
# E. packed operands of the training step (ttsb_repack_batched)
# =====================================================================================================================
def _expected_packs(model, key, ent):
    """The packed operand `key` of TrainEngine.P built on the host with torch ops from the Keras-layout weights."""
    from transformertts_b200.model.models import _round_up
    W = model.weights

    def pad2(x, rows, cols):
        out = torch.zeros(rows, cols, dtype=x.dtype, device=x.device)
        out[:x.shape[0], :x.shape[1]] = x
        return out

    if isinstance(ent, tuple):                               # padded LayerNorm gamma / beta of a predictor conv block
        pre = key                                            # e.g. 'dur_pred.ln0'
        return tuple(pad2(W[f'{pre}.{n}'].view(1, -1), 1, ent[i].numel()).view(-1) for i, n in enumerate(('gamma', 'beta')))
    w_hi = ent.w_hi
    if key.endswith('.d') or key.endswith('.dx') or key.endswith('.da'):   # data-gradient packings [K_pad, N_pad]
        base = key.rsplit('.', 1)[0]
        if key.endswith('.qkv.d'):
            stem = key[:-len('qkv.d')]
            w = torch.cat([W[stem + n + '.w'] for n in ('wq', 'wk', 'wv')], 1)
        elif key.endswith('.wo.dx') or key.endswith('.wo.da'):
            wo = W[base + '.w']
            half = wo.shape[0] // 2
            w = wo[:half] if key.endswith('.dx') else wo[half:]
        else:
            w = W[base + '.w']
        if w.dim() == 3:                                    # Conv1D (k, Cin, Cout): taps side by side, each padded to 64
            k, cin, cout = w.shape
            cpad = _round_up(cout, 64)
            taps = [pad2(w[t].bfloat16(), cin, cpad) for t in range(k)]
            return (pad2(torch.cat(taps, 1), w_hi.shape[0], k * cpad),)
        return (pad2(w.bfloat16(), w_hi.shape[0], _round_up(w.shape[1], 64)),)
    if key.endswith('.qkv'):
        stem = key[:-len('qkv')]
        w = torch.cat([W[stem + n + '.w'] for n in ('wq', 'wk', 'wv')], 1)
        b = torch.cat([W[stem + n + '.b'] for n in ('wq', 'wk', 'wv')])
    else:
        w, b = W[key + '.w'], W[key + '.b']
    w2 = w.reshape(-1, w.shape[-1])
    return (pad2(w2.T.bfloat16(), ent.n_pad, w2.shape[0]), pad2(b.view(1, -1), 1, ent.n_pad).view(-1))


def _packed_tensors(ent):
    return ent if isinstance(ent, tuple) else ((ent.w_hi,) if ent.bias is None else (ent.w_hi, ent.bias))


def _poison_and_compare(eng, model):
    P = eng.P
    keys = [k for k in P if not k.endswith('.pe')]
    for k in keys:
        for t in _packed_tensors(P[k]):
            t.fill_(float('nan'))
    eng._pack()
    torch.cuda.synchronize()
    n = 0
    for k in keys:
        got, want = _packed_tensors(P[k]), _expected_packs(model, k, P[k])
        assert len(got) == len(want), k
        for a, b in zip(got, want):
            assert a.shape == b.shape, (k, a.shape, b.shape)
            iv = torch.int16 if a.dtype == torch.bfloat16 else torch.int32
            assert torch.equal(a.view(iv), b.view(iv)), k
            n += a.numel()
    return keys, n


@pytest.mark.parametrize('cfg_name', ['C1', 'LJ256'])
def test_repacked_training_operands_bit_exact(cfg_name):
    """Every packed operand the training step refreshes with one ttsb_repack_batched launch (forward [N_pad, K] with q|k|v
    stacked, Dense / Conv1D data-gradient packings, bias and LayerNorm vectors), poisoned with NaN and re-packed, equals
    the host-built matrix bit for bit including zero padding -- before and after an Adam step changes the weights."""
    from oracle import forward_oracle as fo
    from transformertts_b200.model.models import ForwardTransformer
    from transformertts_b200.model.training import Adam
    cfg = fo.CONFIGS[cfg_name]
    model = ForwardTransformer(**cfg, train_dropout=False)
    model.set_weights(fo.init_params(cfg, seed=7))
    model._compile(Adam(1e-2))
    eng = model._get_engine()
    eng._pack()
    keys, n = _poison_and_compare(eng, model)
    kinds = {k.rsplit('.', 1)[-1] for k in keys}
    assert {'qkv', 'wo', 'd', 'dx', 'da', 'out'} <= kinds and any('.ln' in k for k in keys), sorted(kinds)
    before = eng.P['out'].w_hi.clone()
    g = torch.Generator(device=DEV).manual_seed(36)
    eng.flat_g.copy_(torch.randn(eng.flat_g.shape, generator=g, device=DEV))
    eng.apply_adam(model.optimizer)
    keys2, n2 = _poison_and_compare(eng, model)
    assert keys2 == keys and n2 == n
    assert not torch.equal(eng.P['out'].w_hi, before)      # the weights did move
    print(f'{cfg_name}: {len(keys)} packed operands, {n} elements bit-exact before and after an Adam step')
