"""Helpers that run the UNMODIFIED reference sources on top of tests/tf_shim, for the scripts under tests/golden/ that
write the golden vectors.  The reference is a checkout of as-ideas/TransformerTTS named by the TTS_REFERENCE environment
variable; the tests themselves only read the committed golden files."""
from __future__ import annotations

import os
import sys
from pathlib import Path

import torch

REFERENCE = Path(os.environ['TTS_REFERENCE']) if os.environ.get('TTS_REFERENCE') else None
SHIM = Path(__file__).resolve().parent / 'tf_shim'


def available() -> bool:
    return REFERENCE is not None and (REFERENCE / 'model' / 'models.py').exists()


def real_tensorflow_available() -> bool:
    """SURVEY 8c probe: is a real TensorFlow importable (never in this image -- there is no wheel)?"""
    import importlib.util
    spec = importlib.util.find_spec('tensorflow')
    return spec is not None and spec.origin is not None and str(SHIM) not in str(spec.origin)


def activate(real_tf: bool = False):
    """Put the reference tree (and, unless real_tf, the shim packages) on sys.path (idempotent)."""
    if not available():
        raise RuntimeError('set TTS_REFERENCE to a checkout of as-ideas/TransformerTTS')
    paths = (str(REFERENCE),) if real_tf else (str(REFERENCE), str(SHIM))
    for p in paths:
        if p in sys.path:
            sys.path.remove(p)
        sys.path.insert(0, p)
    import tensorflow  # noqa: F401
    is_shim = getattr(tensorflow, '__version__', '').endswith('shim')
    assert is_shim != real_tf, 'wrong tensorflow module on sys.path for this mode'


def adam_first_moment(optimizer, var):
    """First-moment slot of `var` (shim Adam keeps (m, v) per variable; real Keras has get_slot)."""
    if hasattr(optimizer, '_slots'):
        return optimizer._slots[id(var)][0]
    return torch.from_numpy(optimizer.get_slot(var, 'm').numpy())


def _assign(var, value):
    value = torch.as_tensor(value).detach().float()
    assert tuple(var.shape) == tuple(value.shape), (tuple(var.shape), tuple(value.shape))
    var.assign(value)


def assign_all(named: dict, params: dict):
    missing = set(named) ^ set(params)
    assert not missing, f'parameter name mismatch: {sorted(missing)[:6]}'
    for k, var in named.items():
        _assign(var, params[k])


def _mha_vars(out, pre, mha):
    for ours, theirs in (('wq', mha.wq), ('wk', mha.wk), ('wv', mha.wv), ('wo', mha.dense)):
        out[pre + ours + '.w'], out[pre + ours + '.b'] = theirs.kernel, theirs.bias


def _self_attention_stack_vars(out, name, stack, n_dense):
    """SelfAttentionBlocks (model/layers.py:267-310): dense blocks first, conv blocks after."""
    out[f'{name}.ln.gamma'], out[f'{name}.ln.beta'] = stack.layernorm.gamma, stack.layernorm.beta
    out[f'{name}.pos_scalar'] = stack.pos_encoding_scalar
    for i, blk in enumerate(list(stack.encoder_SADB) + list(stack.encoder_SACB)):
        pre = f'{name}.b{i}.'
        _mha_vars(out, pre, blk.sarn.mha)
        out[pre + 'ln1.gamma'], out[pre + 'ln1.beta'] = blk.sarn.last_ln.gamma, blk.sarn.last_ln.beta
        if i < n_dense:
            out[pre + 'ffn1.w'], out[pre + 'ffn1.b'] = blk.ffn.d1.kernel, blk.ffn.d1.bias
            out[pre + 'ffn2.w'], out[pre + 'ffn2.b'] = blk.ffn.d2.kernel, blk.ffn.d2.bias
            out[pre + 'ln2.gamma'], out[pre + 'ln2.beta'] = blk.ffn.last_ln.gamma, blk.ffn.last_ln.beta
        else:
            for j, c in enumerate(list(blk.conv.convolutions) + [blk.conv.last_conv]):
                out[pre + f'conv{j}.w'], out[pre + f'conv{j}.b'] = c.kernel, c.bias
            out[pre + 'ln2.gamma'], out[pre + 'ln2.beta'] = blk.conv.normalization.gamma, blk.conv.normalization.beta


def ft_named_parameters(model, cfg: dict) -> dict:
    """{flat parameter name of transformertts_b200/model/models.py: the reference ForwardTransformer's Variable}."""
    out = {'embedding': model.encoder_prenet.embeddings}
    _self_attention_stack_vars(out, 'encoder', model.encoder, int(cfg['encoder_dense_blocks']))
    _self_attention_stack_vars(out, 'decoder', model.decoder, int(cfg['decoder_dense_blocks']))
    for name, pred in (('dur_pred', model.dur_pred), ('pitch_pred', model.pitch_pred)):
        for j, c in enumerate(list(pred.conv_blocks.convolutions) + [pred.conv_blocks.last_conv]):
            out[f'{name}.conv{j}.w'], out[f'{name}.conv{j}.b'] = c.kernel, c.bias
            ln = pred.conv_blocks.normalization[j]
            out[f'{name}.ln{j}.gamma'], out[f'{name}.ln{j}.beta'] = ln.gamma, ln.beta
        out[f'{name}.out.w'], out[f'{name}.out.b'] = pred.linear.kernel, pred.linear.bias
    out['pitch_embed.w'], out['pitch_embed.b'] = model.pitch_embed.kernel, model.pitch_embed.bias
    out['out.w'], out['out.b'] = model.out.kernel, model.out.bias
    return out


def aligner_named_parameters(model, cfg: dict) -> dict:
    """{flat parameter name of transformertts_b200/model/aligner.py: the reference Aligner's Variable}."""
    out = {'embedding': model.encoder_prenet.embeddings}
    _self_attention_stack_vars(out, 'encoder', model.encoder, len(cfg['encoder_num_heads']))
    out['prenet.d1.w'], out['prenet.d1.b'] = model.decoder_prenet.d1.kernel, model.decoder_prenet.d1.bias
    out['prenet.d2.w'], out['prenet.d2.b'] = model.decoder_prenet.d2.kernel, model.decoder_prenet.d2.bias
    dec = model.decoder
    out['decoder.ln.gamma'], out['decoder.ln.beta'] = dec.layernorm.gamma, dec.layernorm.beta
    out['decoder.pos_scalar'] = dec.pos_encoding_scalar
    for i, blk in enumerate(list(dec.CADB) + [dec.last_CADB]):
        pre = f'decoder.b{i}.'
        _mha_vars(out, pre + 'sa.', blk.sarn.mha)
        out[pre + 'sa.ln.gamma'], out[pre + 'sa.ln.beta'] = blk.sarn.last_ln.gamma, blk.sarn.last_ln.beta
        _mha_vars(out, pre + 'ca.', blk.carn.mha)
        out[pre + 'ca.ln.gamma'], out[pre + 'ca.ln.beta'] = blk.carn.layernorm.gamma, blk.carn.layernorm.beta
        out[pre + 'ffn1.w'], out[pre + 'ffn1.b'] = blk.ffn.d1.kernel, blk.ffn.d1.bias
        out[pre + 'ffn2.w'], out[pre + 'ffn2.b'] = blk.ffn.d2.kernel, blk.ffn.d2.bias
        out[pre + 'ln2.gamma'], out[pre + 'ln2.beta'] = blk.ffn.last_ln.gamma, blk.ffn.last_ln.beta
    out['final_proj.w'], out['final_proj.b'] = model.final_proj_mel.kernel, model.final_proj_mel.bias
    out['postnet.stop.w'], out['postnet.stop.b'] = model.decoder_postnet.stop_linear.kernel, model.decoder_postnet.stop_linear.bias
    out['postnet.mel.w'], out['postnet.mel.b'] = model.decoder_postnet.mel_out.kernel, model.decoder_postnet.mel_out.bias
    return out


def reference_forward_transformer(cfg: dict, params: dict, warm_inputs, **overrides):
    """Instantiate the reference's model/models.py:ForwardTransformer (unmodified) under the shim with `params`.
    `warm_inputs` = (tokens, durations (B,Tp,1), pitch (B,Tp,1)): one throw-away call creates the Keras variables (the
    reference's own build_model_weights() feeds a 1x1 dummy, which produces an empty decoder input)."""
    activate()
    from model.models import ForwardTransformer  # the reference class
    kw = dict(cfg)
    kw.setdefault('phoneme_language', 'en-us')
    kw.setdefault('with_stress', False)
    kw.setdefault('model_breathing', False)
    kw.setdefault('transposed_attn_convs', True)
    kw.update(overrides)
    kw['debug'] = True
    model = ForwardTransformer(**kw)
    tok, dur, pit = warm_inputs
    with torch.no_grad():
        model.call(tok, target_durations=dur, target_pitch=pit, training=False)
    assign_all(ft_named_parameters(model, cfg), params)
    return model


def reference_aligner(cfg: dict, params: dict, warm_inputs, **overrides):
    """Instantiate the reference's model/models.py:Aligner (unmodified) under the shim with `params`."""
    activate()
    from model.models import Aligner  # the reference class
    kw = {k: v for k, v in cfg.items() if k not in ('vocab_size', 'stop_loss_scaling')}
    kw.update(overrides)
    kw['debug'] = True
    model = Aligner(**kw)
    assert model.text_pipeline.tokenizer.vocab_size == int(cfg['vocab_size'])
    tok, mel = warm_inputs
    with torch.no_grad():
        model.call(tok, mel, training=False)
    assign_all(aligner_named_parameters(model, cfg), params)
    return model
