"""CPU oracle for the ForwardTransformer text->mel hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` may be imported by the product
package ``transformertts_b200``; only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` use it, and only as the
checker / reported CPU baseline.

PARITY STATUS: the reference's arithmetic lives in TensorFlow/Keras (``tensorflow>=2.2.0``, ``requirements.txt:7``), which
is not installed here and cannot be installed (no network), and the reference's own tests hold no golden vectors for this
path (SURVEY.md section 4).  This restatement is pinned to the REFERENCE'S OWN CODE instead: tests/golden/make_reference_pins.py
imports the unmodified model/{layers,models,transformer_utils}.py and utils/losses.py of the reference, runs them on
tests/tf_shim (a torch-backed stand-in for the TensorFlow/Keras primitives, semantics from the TF documentation; the
reference's tests/test_loss.py known answers pass on it), and tests/test_reference_shim.py compares ``ForwardTransformer.call`` / ``predict`` / ``_train_step``
(loss, every gradient, Keras Adam) with this file on C1 / LJ256 / LJ256-dense / REF384: agreement 2e-5 (mel), 1e-5 (attention),
bit-exact masks and integer durations.  The golden vectors tests/golden/{c1_forward,ref_lj256,ref_train_c1}.npz are written by
those reference-code runs (tests/golden/make_golden_ref.py; make_golden_tf.py does the same on a machine with real TensorFlow).
What remains unpinned is the primitive layer of the shim itself (documented TF behaviour, not TF binaries).  Also kept:
  * the ``Expand`` docstring example (``model/layers.py:532-542``) -- tests/test_oracle.py
  * an independent second implementation built from stock ``torch.nn.functional`` ops -- tests/test_oracle.py

Every function cites the reference lines it restates (paths relative to the reference
repo root).  All math is torch-CPU; ``dtype`` is float32 (the reference's type) unless a
float64 "truth" run is requested.  Keras layouts are kept: Dense kernel (in, out), Conv1D
kernel (k, in, out), activations (B, T, C).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import numpy as np
import torch

Tensor = torch.Tensor
LN_EPS = 1e-6  # model/layers.py:27,96,207,295,508
NEG_MASK = -1e9  # model/layers.py:187
VOCAB_SIZE = 127  # 126 symbols + pad id 0 (data/text/tokenizer.py:17-20, symbols.py:12)


# ----------------------------------------------------------------------------------------
# model/transformer_utils.py
# ----------------------------------------------------------------------------------------
def positional_encoding(position: int, model_dim: int) -> Tensor:
    """model/transformer_utils.py:5-21 -- table built in float64, cast to float32."""
    pos = np.arange(position)[:, np.newaxis]
    i = np.arange(model_dim)[np.newaxis, :]
    angle_rates = 1 / np.power(10000, (2 * (i // 2)) / np.float32(model_dim))
    angle_rads = pos * angle_rates
    angle_rads[:, 0::2] = np.sin(angle_rads[:, 0::2])
    angle_rads[:, 1::2] = np.cos(angle_rads[:, 1::2])
    return torch.from_numpy(angle_rads[np.newaxis, ...].astype(np.float32))


def create_encoder_padding_mask(seq: Tensor) -> Tensor:
    """model/transformer_utils.py:24-26 -- (B,1,1,T) float, 1.0 where token id == 0."""
    return (seq == 0).to(torch.float32)[:, None, None, :]


def create_mel_padding_mask(seq: Tensor) -> Tensor:
    """model/transformer_utils.py:29-32 -- value-derived: frame is padding iff sum|x| == 0."""
    s = seq.abs().sum(dim=-1)
    return (s == 0).to(torch.float32)[:, None, None, :]


# ----------------------------------------------------------------------------------------
# Keras primitives (third-party semantics, SURVEY App. A.10)
# ----------------------------------------------------------------------------------------
def layer_norm(x: Tensor, gamma: Tensor, beta: Tensor, eps: float = LN_EPS) -> Tensor:
    """keras LayerNormalization(axis=-1, epsilon=1e-6), non-fused path: biased variance,
    y = (x-mean)*rsqrt(var+eps)*gamma + beta."""
    mean = x.mean(dim=-1, keepdim=True)
    var = ((x - mean) ** 2).mean(dim=-1, keepdim=True)
    inv = torch.rsqrt(var + eps)
    return (x - mean) * inv * gamma + beta


# ----------------------------------------------------------------------------------------
# bf16-operand emulation (test infrastructure for the TRAINING step): the CUDA path feeds every tensor-core product with
# bf16-rounded operands, forward and backward (activations, weights and incoming gradients are rounded once, accumulation
# is fp32).  With EMULATE_BF16 set, every matrix product of this oracle does the same, so that a comparison with the GPU
# gradients sees only summation-order noise plus the few roundings that are not operand roundings (saved probabilities),
# not the ~10 % per-tensor bf16 noise that would hide a wrong small term.  Off by default: the oracle is the fp32 reference.
# ----------------------------------------------------------------------------------------
EMULATE_BF16 = False


def _r16(t: Tensor) -> Tensor:
    return t.to(torch.bfloat16).to(t.dtype)


class _Bf16MatMul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        a16, b16 = _r16(a), _r16(b)
        ctx.save_for_backward(a16, b16)
        return a16 @ b16

    @staticmethod
    def backward(ctx, g):
        a16, b16 = ctx.saved_tensors
        g16 = _r16(g)
        ga = g16 @ b16.transpose(-1, -2)
        gb = a16.transpose(-1, -2) @ g16
        while gb.dim() > b16.dim():      # a (.., M, K) @ b (K, N): the weight gradient sums over the leading dimensions
            gb = gb.sum(0)
        return ga, gb


def mm(a: Tensor, b: Tensor) -> Tensor:
    """a @ b, with bf16-rounded operands (forward and backward) under EMULATE_BF16."""
    if EMULATE_BF16:
        if b.dim() == 2 and a.dim() > 2:
            return _Bf16MatMul.apply(a.reshape(-1, a.shape[-1]), b).reshape(*a.shape[:-1], b.shape[-1])
        return _Bf16MatMul.apply(a, b)
    return a @ b


def dense(x: Tensor, w: Tensor, b: Tensor, act: Optional[str] = None) -> Tensor:
    y = mm(x, w) + b
    if act == 'relu':
        y = torch.relu(y)
    return y


def conv1d_same(x: Tensor, w: Tensor, b: Tensor) -> Tensor:
    """keras Conv1D(padding='same', stride 1), channels-last.  x (B,T,Cin), w (k,Cin,Cout).
    y[b,t] = b + sum_j x[b, t + j - (k-1)//2] @ w[j], zero outside [0,T)."""
    k = w.shape[0]
    B, T, _ = x.shape
    left = (k - 1) // 2
    y = torch.zeros(B, T, w.shape[2], dtype=x.dtype) + b
    for j in range(k):
        s = j - left  # input offset
        lo, hi = max(0, -s), min(T, T - s)
        if hi > lo:
            y[:, lo:hi] += mm(x[:, lo + s:hi + s], w[j])
    return y


def dropout(x: Tensor, rate: float, training: bool, gen: Optional[torch.Generator]) -> Tensor:
    """keras Dropout: inverted scaling, identity at inference."""
    if not training or rate <= 0.0:
        return x
    keep = (torch.rand(x.shape, generator=gen) >= rate).to(x.dtype)
    return x * keep / (1.0 - rate)


# ----------------------------------------------------------------------------------------
# model/layers.py
# ----------------------------------------------------------------------------------------
def multi_head_attention(p: Dict[str, Tensor], pre: str, v: Tensor, k: Tensor, q_in: Tensor, mask: Tensor,
                         num_heads: int, rate: float, training: bool, gen) -> (Tensor, Tensor):
    """model/layers.py:105-151 (MHA) and :154-195 (scaled dot product)."""
    B, Tq, d = q_in.shape
    depth = d // num_heads
    q = dense(q_in, p[pre + 'wq.w'], p[pre + 'wq.b'])
    kk = dense(k, p[pre + 'wk.w'], p[pre + 'wk.b'])
    vv = dense(v, p[pre + 'wv.w'], p[pre + 'wv.b'])

    def split(t):
        return t.reshape(B, -1, num_heads, depth).permute(0, 2, 1, 3)

    q, kk, vv = split(q), split(kk), split(vv)
    logits = mm(q, kk.transpose(-1, -2))
    logits = logits / math.sqrt(float(depth))
    if mask is not None:
        logits = logits + mask.to(logits.dtype) * NEG_MASK
    weights = torch.softmax(logits, dim=-1)
    weights = dropout(weights, rate, training, gen)
    out = mm(weights, vv)
    out = out.permute(0, 2, 1, 3).reshape(B, Tq, d)
    concat_query = torch.cat([q_in, out], dim=-1)  # layers.py:148 -- (B,T,2d)
    output = dense(concat_query, p[pre + 'wo.w'], p[pre + 'wo.b'])
    output = dropout(output, rate, training, gen)
    return output, weights


def self_attention_block(p, pre, x, mask4, kind, num_heads, rate, training, gen):
    """SelfAttentionResNorm (:198-211) + SelfAttentionDenseBlock (:214-230) or
    SelfAttentionConvBlock (:233-264) with CNNResNorm (:6-40; the Transposed variant :43-79
    permutes with the identity permutation and is numerically the same)."""
    attn_out, w = multi_head_attention(p, pre, x, x, x, mask4, num_heads, rate, training, gen)
    y = layer_norm(attn_out + x, p[pre + 'ln1.gamma'], p[pre + 'ln1.beta'])
    keep = 1.0 - mask4[:, 0, 0, :, None].to(x.dtype)
    y = y * keep
    if kind == 'dense':
        h = dense(y, p[pre + 'ffn1.w'], p[pre + 'ffn1.b'], 'relu')
        h = dense(h, p[pre + 'ffn2.w'], p[pre + 'ffn2.b'])
        h = dropout(h, rate, training, gen)
        z = layer_norm(h + y, p[pre + 'ln2.gamma'], p[pre + 'ln2.beta'])
    else:
        n_conv = sum(1 for key in p if key.startswith(pre + 'conv') and key.endswith('.w'))
        h = y
        for j in range(n_conv - 1):
            h = torch.relu(conv1d_same(h, p[pre + f'conv{j}.w'], p[pre + f'conv{j}.b']))
        h = conv1d_same(h, p[pre + f'conv{n_conv - 1}.w'], p[pre + f'conv{n_conv - 1}.b'])
        h = dropout(h, rate, training, gen)
        z = layer_norm(y + h, p[pre + 'ln2.gamma'], p[pre + 'ln2.beta'])
    return z * keep, w


def self_attention_blocks(p, name, cfg_stack, inputs, mask4, training, gen):
    """model/layers.py:267-310.  LN(inputs) first, then + scalar*PE, dropout, blocks."""
    T = inputs.shape[1]
    x = layer_norm(inputs, p[f'{name}.ln.gamma'], p[f'{name}.ln.beta'])
    pe = cfg_stack['pe'][:, :T, :].to(x.dtype)
    x = x + p[f'{name}.pos_scalar'] * pe
    x = dropout(x, cfg_stack['dropout'], training, gen)
    attn = {}
    cname = name.capitalize()
    n_dense = cfg_stack['dense_blocks']
    for i, nh in enumerate(cfg_stack['num_heads']):
        kind = 'dense' if i < n_dense else 'conv'
        x, w = self_attention_block(p, f'{name}.b{i}.', x, mask4, kind, nh, cfg_stack['dropout'], training, gen)
        if kind == 'dense':
            attn[f'{cname}_DenseBlock{i + 1}_SelfAttention'] = w
        else:
            attn[f'{cname}_ConvBlock{i - n_dense + 1}_SelfAttention'] = w
    return x, attn


def stat_predictor(p, pre, x, mask, n_layers, dense_act, rate, training, gen):
    """StatPredictor (:463-485) over CNNDropout (:488-524): x*mask -> [conv->relu->LN->dropout]*n
    -> Dense(1, act) -> *mask."""
    x = x * mask
    for j in range(n_layers):
        x = torch.relu(conv1d_same(x, p[pre + f'conv{j}.w'], p[pre + f'conv{j}.b']))
        x = layer_norm(x, p[pre + f'ln{j}.gamma'], p[pre + f'ln{j}.beta'])
        x = dropout(x, rate, training, gen)
    x = dense(x, p[pre + 'out.w'], p[pre + 'out.b'], 'relu' if dense_act == 'relu' else None)
    return x * mask


def expand(x: Tensor, dimensions: Tensor) -> Tensor:
    """model/layers.py:549-565, followed step by step (tile x max_dur -> mask -> boolean_mask ->
    ragged -> dense).  dimensions: (B,Tp,1) float or int."""
    dims = torch.round(dimensions.squeeze(-1).to(torch.float64)).to(torch.int32)  # tf.math.round: half-to-even
    B, Tp, d = x.shape
    if (dims < 0).any():
        raise ValueError('negative duration')
    max_dim = int(dims.max()) if dims.numel() else 0
    # RaggedTensor.from_row_lengths(ones(tot), dims.flatten()).to_tensor(): (B*Tp, max_dim)
    index_masks = (torch.arange(max_dim)[None, :] < dims.reshape(-1, 1)).to(torch.float32)
    index_masks = index_masks.reshape(B, Tp * max_dim)
    non_zeros = Tp * max_dim - (max_dim - dims).sum(dim=1)
    tiled = x.repeat(1, 1, max_dim)  # tf.tile(x, [1,1,max_dim])
    reshaped = tiled.reshape(B, Tp * max_dim, d)
    mask_reshape = reshaped * index_masks[:, :, None].to(x.dtype)
    flat = mask_reshape[index_masks > 0]  # (tot, d), row-major order
    T_out = int(non_zeros.max()) if B else 0
    out = torch.zeros(B, T_out, d, dtype=x.dtype)
    off = 0
    for b in range(B):
        n = int(non_zeros[b])
        out[b, :n] = flat[off:off + n]
        off += n
    return out


def round_durations(dimensions: Tensor) -> Tensor:
    """model/layers.py:550-551 -- tf.cast(tf.math.round(x), int32) (round-half-to-even)."""
    return torch.round(dimensions.squeeze(-1).to(torch.float32)).to(torch.int32)


def expand_indices(int_durations: Tensor):
    """Integer view of Expand: per-row output lengths and, for each output frame, the phoneme index it
    copies (-1 at padded frames).  Bit-exact target for the CUDA length regulator."""
    B, Tp = int_durations.shape
    lengths = int_durations.sum(dim=1).to(torch.int32)
    Tm = int(lengths.max()) if B else 0
    idx = torch.full((B, Tm), -1, dtype=torch.int32)
    for b in range(B):
        r = torch.repeat_interleave(torch.arange(Tp, dtype=torch.int32), int_durations[b].to(torch.int64))
        idx[b, :r.numel()] = r
    return lengths, idx


# ----------------------------------------------------------------------------------------
# model/models.py -- ForwardTransformer
# ----------------------------------------------------------------------------------------
def normalize_config(cfg: dict) -> dict:
    """Pick the constructor arguments of ForwardTransformer (model/models.py:345-372)."""
    c = dict(cfg)
    c.setdefault('mel_channels', 80)
    c.setdefault('dropout_rate', 0.1)
    c.setdefault('predictors_dropout', 0.1)
    c.setdefault('vocab_size', VOCAB_SIZE)
    return c


def stack_cfg(cfg: dict, which: str) -> dict:
    return {
        'num_heads': list(cfg[f'{which}_num_heads']),
        'dense_blocks': int(cfg[f'{which}_dense_blocks']),
        'dropout': float(cfg['dropout_rate']),
        'pe': positional_encoding(int(cfg[f'{which}_max_position_encoding']), int(cfg[f'{which}_model_dimension'])),
    }


def forward_transformer_call(p: Dict[str, Tensor], cfg: dict, x: Tensor,
                             target_durations: Optional[Tensor] = None,
                             target_pitch: Optional[Tensor] = None,
                             training: bool = False,
                             durations_scalar: float = 1.0,
                             max_durations_mask: Optional[Tensor] = None,
                             min_durations_mask: Optional[Tensor] = None,
                             gen: Optional[torch.Generator] = None,
                             _cache: Optional[dict] = None) -> dict:
    """model/models.py:518-550.  x int (B,Tp); targets (B,Tp,1)."""
    cfg = normalize_config(cfg)
    dt = p['embedding'].dtype
    if _cache is None:
        _cache = {}
    if 'enc' not in _cache:
        _cache['enc'] = stack_cfg(cfg, 'encoder')
        _cache['dec'] = stack_cfg(cfg, 'decoder')
    enc_mask = create_encoder_padding_mask(x)
    h = p['embedding'][x.long()]
    h, enc_attn = self_attention_blocks(p, 'encoder', _cache['enc'], h, enc_mask, training, gen)
    padding_mask = 1.0 - enc_mask[:, 0, 0, :, None].to(dt)
    n_dur = len(cfg['duration_conv_filters'])
    n_pit = len(cfg['pitch_conv_filters'])
    durations = stat_predictor(p, 'dur_pred.', h, padding_mask, n_dur, 'relu', cfg['predictors_dropout'], training, gen)
    pitch = stat_predictor(p, 'pitch_pred.', h, padding_mask, n_pit, 'linear', cfg['predictors_dropout'], training, gen)
    src_pitch = target_pitch.to(dt) if target_pitch is not None else pitch
    pitch_embed = dense(src_pitch, p['pitch_embed.w'], p['pitch_embed.b'], 'relu')
    h = h + pitch_embed
    if target_durations is not None:
        use_durations = target_durations
    else:
        use_durations = durations * durations_scalar
    if max_durations_mask is not None:
        use_durations = torch.minimum(use_durations.to(dt), max_durations_mask.to(dt)[..., None])
    if min_durations_mask is not None:
        use_durations = torch.maximum(use_durations.to(dt), min_durations_mask.to(dt)[..., None])
    mels = expand(h, use_durations)
    expanded_mask = create_mel_padding_mask(mels)
    mels, dec_attn = self_attention_blocks(p, 'decoder', _cache['dec'], mels, expanded_mask, training, gen)
    mels = dense(mels, p['out.w'], p['out.b'])
    return {'mel': mels, 'duration': durations, 'pitch': pitch, 'expanded_mask': expanded_mask,
            'encoder_attention': enc_attn, 'decoder_attention': dec_attn,
            'int_durations': round_durations(use_durations)}


def predict(p, cfg, inp: Tensor, speed_regulator: float = 1.0, phoneme_durations=None, phoneme_pitch=None,
            max_durations_mask=None, min_durations_mask=None) -> dict:
    """model/models.py:559-577 with encode=False.  The reference overwrites passed max/min masks with the
    dict-derived ones (:567-568): +inf / 0 when no per-phoneme dict is given."""
    if inp.dim() < 2:
        inp = inp[None]
    inp = inp.to(torch.int32)
    dur_scalar = float(np.float32(1.0 / speed_regulator))
    max_mask = torch.full(inp.shape, float('inf')) if max_durations_mask is None else max_durations_mask
    min_mask = torch.zeros(inp.shape) if min_durations_mask is None else min_durations_mask
    out = forward_transformer_call(p, cfg, inp, phoneme_durations, phoneme_pitch, False, dur_scalar, max_mask, min_mask)
    out['mel'] = out['mel'].squeeze()
    return out


# ----------------------------------------------------------------------------------------
# utils/losses.py + train step
# ----------------------------------------------------------------------------------------
def masked_mean_absolute_error(targets: Tensor, pred: Tensor) -> Tensor:
    """utils/losses.py:41-49 as called from weighted_sum_losses (:63-70): mask=None, so the mask branch is
    skipped and the result is the plain mean over ALL elements (padding included)."""
    return (targets.to(pred.dtype) - pred).abs().mean()


def weighted_sum_losses(targets, pred, coeffs=(1.0, 1.0, 3.0)):
    """utils/losses.py:63-70 with the weights of model/models.py:485."""
    vals = [masked_mean_absolute_error(t, q) for t, q in zip(targets, pred)]
    total = sum(c * v for c, v in zip(coeffs, vals))
    return total, vals


def loss_from_batch(p, cfg, phonemes, mel_tgt, dur_tgt, pitch_tgt, training=True, gen=None):
    """model/models.py:464-479 (forward + loss part of _train_step / _val_step)."""
    td = dur_tgt[..., None]
    tp = pitch_tgt[..., None]
    mel_len = mel_tgt.shape[1]
    out = forward_transformer_call(p, cfg, phonemes, td, tp, training=training, gen=gen)
    loss, vals = weighted_sum_losses((mel_tgt, td, tp), (out['mel'][:, :mel_len, :], out['duration'], out['pitch']))
    out['loss'] = loss
    out['losses'] = {'mel': vals[0], 'duration': vals[1], 'pitch': vals[2]}
    return out


def adam_tf_step(param: Tensor, grad: Tensor, m: Tensor, v: Tensor, step: int, lr: float,
                 beta1: float = 0.9, beta2: float = 0.98, eps: float = 1e-9):
    """Keras (TF 2.2-era) Adam, utils/training_config_manager.py:102-106:
    lr_t = lr*sqrt(1-b2^t)/(1-b1^t); theta -= lr_t * m / (sqrt(v) + eps)   (eps outside the correction)."""
    m.mul_(beta1).add_(grad, alpha=1 - beta1)
    v.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    lr_t = lr * math.sqrt(1 - beta2 ** step) / (1 - beta1 ** step)
    param.sub_(lr_t * m / (v.sqrt() + eps))


# ----------------------------------------------------------------------------------------
# Seeded parameter / input generators (SURVEY 8d "weights (all)")
# ----------------------------------------------------------------------------------------
def _glorot(gen, shape, fan_in, fan_out):
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return (torch.rand(shape, generator=gen) * 2 - 1) * lim


def init_params(cfg: dict, seed: int = 7, dtype=torch.float32) -> Dict[str, Tensor]:
    """Glorot-uniform kernels, non-zero biases (0.05*N), LN gamma 1+0.1*N / beta 0.1*N, embedding U(-.05,.05),
    pos_scalar 0.8 (encoder) / 1.1 (decoder).  Non-default biases/LN so every bias path is exercised."""
    cfg = normalize_config(cfg)
    g = torch.Generator(device='cpu').manual_seed(seed)
    p: Dict[str, Tensor] = {}
    d_enc, d_dec = int(cfg['encoder_model_dimension']), int(cfg['decoder_model_dimension'])

    def bias(n):
        return 0.05 * torch.randn(n, generator=g)

    def ln(prefix, n):
        p[prefix + '.gamma'] = 1.0 + 0.1 * torch.randn(n, generator=g)
        p[prefix + '.beta'] = 0.1 * torch.randn(n, generator=g)

    def lin(prefix, fin, fout):
        p[prefix + '.w'] = _glorot(g, (fin, fout), fin, fout)
        p[prefix + '.b'] = bias(fout)

    def conv(prefix, k, cin, cout):
        p[prefix + '.w'] = _glorot(g, (k, cin, cout), k * cin, k * cout)
        p[prefix + '.b'] = bias(cout)

    p['embedding'] = (torch.rand((cfg['vocab_size'], d_enc), generator=g) * 2 - 1) * 0.05
    for name, d, scalar in (('encoder', d_enc, 0.8), ('decoder', d_dec, 1.1)):
        ln(f'{name}.ln', d)
        p[f'{name}.pos_scalar'] = torch.tensor(scalar)
        n_dense = int(cfg[f'{name}_dense_blocks'])
        for i, _nh in enumerate(cfg[f'{name}_num_heads']):
            pre = f'{name}.b{i}.'
            lin(pre + 'wq', d, d)
            lin(pre + 'wk', d, d)
            lin(pre + 'wv', d, d)
            lin(pre + 'wo', 2 * d, d)
            ln(pre + 'ln1', d)
            if i < n_dense:
                F = int(cfg[f'{name}_feed_forward_dimension'])
                lin(pre + 'ffn1', d, F)
                lin(pre + 'ffn2', F, d)
            else:
                k = int(cfg[f'{name}_attention_conv_kernel'])
                cin = d
                for j, f in enumerate(cfg[f'{name}_attention_conv_filters']):
                    conv(pre + f'conv{j}', k, cin, int(f))
                    cin = int(f)
            ln(pre + 'ln2', d)
    for name, filt, k in (('dur_pred', cfg['duration_conv_filters'], cfg['duration_kernel_size']),
                          ('pitch_pred', cfg['pitch_conv_filters'], cfg['pitch_kernel_size'])):
        cin = d_enc
        for j, f in enumerate(filt):
            conv(f'{name}.conv{j}', int(k), cin, int(f))
            ln(f'{name}.ln{j}', int(f))
            cin = int(f)
        lin(f'{name}.out', cin, 1)
    lin('pitch_embed', 1, d_enc)
    lin('out', d_dec, int(cfg['mel_channels']))
    return {k: v.to(dtype) for k, v in p.items()}


CONFIGS = {
    # BASELINE.json configs[0] (C1): 2+2 layers, d=128, one dense + one conv block per stack
    'C1': dict(encoder_model_dimension=128, decoder_model_dimension=128, dropout_rate=0.1,
               encoder_num_heads=[2, 2], decoder_num_heads=[2, 2],
               encoder_max_position_encoding=2000, decoder_max_position_encoding=10000,
               encoder_dense_blocks=1, decoder_dense_blocks=1,
               encoder_feed_forward_dimension=512, decoder_feed_forward_dimension=512,
               encoder_attention_conv_filters=[512, 128], decoder_attention_conv_filters=[512, 128],
               encoder_attention_conv_kernel=3, decoder_attention_conv_kernel=3,
               duration_conv_filters=[256, 226], pitch_conv_filters=[256, 226],
               duration_kernel_size=3, pitch_kernel_size=3, predictors_dropout=0.1, mel_channels=80,
               phoneme_language='en-us', with_stress=True, model_breathing=False, transposed_attn_convs=True),
    # BASELINE.json configs[1]/[2] (C2/C3): LJSpeech ForwardTransformer 6+6, d=256 (SURVEY 8 "LJ256")
    'LJ256': dict(encoder_model_dimension=256, decoder_model_dimension=256, dropout_rate=0.1,
                  encoder_num_heads=[2] * 6, decoder_num_heads=[2] * 6,
                  encoder_max_position_encoding=2000, decoder_max_position_encoding=10000,
                  encoder_dense_blocks=0, decoder_dense_blocks=0,
                  encoder_feed_forward_dimension=None, decoder_feed_forward_dimension=None,
                  encoder_attention_conv_filters=[1024, 256], decoder_attention_conv_filters=[1024, 256],
                  encoder_attention_conv_kernel=3, decoder_attention_conv_kernel=3,
                  duration_conv_filters=[256, 226], pitch_conv_filters=[256, 226],
                  duration_kernel_size=3, pitch_kernel_size=3, predictors_dropout=0.1, mel_channels=80,
                  phoneme_language='en-us', with_stress=True, model_breathing=False, transposed_attn_convs=True),
}
# the yaml as shipped by the reference (config/training_config.yaml:102-124): d=384, 2 heads of 192, conv [1536, 384]
CONFIGS['REF384'] = dict(CONFIGS['LJ256'], encoder_model_dimension=384, decoder_model_dimension=384,
                         encoder_attention_conv_filters=[1536, 384], decoder_attention_conv_filters=[1536, 384])
CONFIGS['LJ256-dense'] = dict(CONFIGS['LJ256'], encoder_dense_blocks=6, decoder_dense_blocks=6,
                              encoder_feed_forward_dimension=1024, decoder_feed_forward_dimension=1024)


def make_inputs(kind: str, B: int, Tp: int, Tm: int, seed: int):
    """Synthetic LJSpeech-shaped batches (SURVEY 8d).  kind 'full': every row Tp tokens, durations sum to Tm
    exactly; kind 'ragged': per-row token / frame counts vary, pad id 0 / duration 0 / pitch 0."""
    g = torch.Generator(device='cpu').manual_seed(seed)
    tokens = torch.zeros(B, Tp, dtype=torch.int32)
    durs = torch.zeros(B, Tp, dtype=torch.int32)
    pitch = torch.zeros(B, Tp)
    for b in range(B):
        if kind == 'full' or b == 0:
            tp_b, tm_b = Tp, Tm
        else:
            tp_b = int(torch.randint(Tp // 2, Tp + 1, (1,), generator=g))
            tm_b = int(torch.randint(Tm // 2, Tm + 1, (1,), generator=g))
        tm_b = max(tm_b, tp_b)
        tokens[b, :tp_b] = torch.randint(1, VOCAB_SIZE, (tp_b,), generator=g, dtype=torch.int32)
        # 1 + multinomial(tm_b - tp_b) composition
        extra = tm_b - tp_b
        w = torch.rand(tp_b, generator=g) + 0.05
        cnt = torch.bincount(torch.multinomial(w, extra, replacement=True, generator=g), minlength=tp_b) if extra > 0 \
            else torch.zeros(tp_b, dtype=torch.int64)
        durs[b, :tp_b] = (1 + cnt).to(torch.int32)
        pitch[b, :tp_b] = torch.randn(tp_b, generator=g)
    return tokens, durs, pitch


def make_mel_targets(durs: Tensor, mel_channels: int, seed: int) -> Tensor:
    g = torch.Generator(device='cpu').manual_seed(seed)
    lengths = durs.sum(dim=1)
    B, Tm = durs.shape[0], int(lengths.max())
    mel = (torch.randn(B, Tm, mel_channels, generator=g) * 2 - 5).clamp(-11.5, 2.0)
    for b in range(B):
        mel[b, int(lengths[b]):] = 0
    return mel


def forward_flops(cfg: dict, tp_lens: List[int], tm_lens: List[int]) -> float:
    """Algorithmic FLOPs of one forward pass over valid tokens only (SURVEY 8d formula)."""
    cfg = normalize_config(cfg)
    total = 0.0
    for name, lens in (('encoder', tp_lens), ('decoder', tm_lens)):
        d = int(cfg[f'{name}_model_dimension'])
        n_dense = int(cfg[f'{name}_dense_blocks'])
        for i, _ in enumerate(cfg[f'{name}_num_heads']):
            for T in lens:
                total += 10 * T * d * d + 4 * T * T * d
                if i < n_dense:
                    total += 4 * T * d * int(cfg[f'{name}_feed_forward_dimension'])
                else:
                    k = int(cfg[f'{name}_attention_conv_kernel'])
                    cin = d
                    for f in cfg[f'{name}_attention_conv_filters']:
                        total += 2 * k * T * cin * int(f)
                        cin = int(f)
    d = int(cfg['encoder_model_dimension'])
    for filt, k in ((cfg['duration_conv_filters'], cfg['duration_kernel_size']),
                    (cfg['pitch_conv_filters'], cfg['pitch_kernel_size'])):
        for T in tp_lens:
            cin = d
            for f in filt:
                total += 2 * int(k) * T * cin * int(f)
                cin = int(f)
            total += 2 * T * cin
    total += sum(2 * T * d for T in tp_lens)
    total += sum(2 * T * int(cfg['decoder_model_dimension']) * int(cfg['mel_channels']) for T in tm_lens)
    return total


def loss_and_grads(p: Dict[str, Tensor], cfg: dict, phonemes, mel_tgt, dur_tgt, pitch_tgt, emulate_bf16: bool = False):
    """Forward (dropout off) + backward with torch autograd on the restated graph: the oracle of the hand-written
    backward pass.  Returns (outputs, {name: grad}).  emulate_bf16: see EMULATE_BF16 above."""
    global EMULATE_BF16
    q = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
    saved, EMULATE_BF16 = EMULATE_BF16, bool(emulate_bf16)
    try:
        out = loss_from_batch(q, cfg, phonemes, mel_tgt, dur_tgt, pitch_tgt, training=False)
        out['loss'].backward()
    finally:
        EMULATE_BF16 = saved
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in q.items()}
    return out, grads
