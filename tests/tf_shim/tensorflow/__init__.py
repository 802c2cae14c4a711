"""Test-only TensorFlow shim on torch CPU tensors (see tests/tf_shim/README.md).

Implements exactly the TF 2.x / Keras entry points the reference's text->mel path uses, with the semantics of the TF
documentation, so that the UNMODIFIED files of the reference can be imported and executed.  Tensors are plain
``torch.Tensor``; ``tf.Variable`` is a ``torch.nn.Parameter`` subclass; ``tf.GradientTape`` is torch autograd.

Known deviations (none on the ForwardTransformer path): ``int / int`` is float32 true division here, float64 in TF
(only ``utils/metrics.diagonal_mask`` of the Aligner divides integer tensors; the result is cast to float32 there).
"""
from __future__ import annotations

import builtins as _b
import math as _math
import types as _types

import numpy as _np
import torch as _torch

__version__ = '2.x-shim'

# ----------------------------------------------------------------------------------------------------------------------
# dtypes / basic aliases
# ----------------------------------------------------------------------------------------------------------------------
float32 = _torch.float32
float64 = _torch.float64
int32 = _torch.int32
int64 = _torch.int64
bool = _torch.bool  # noqa: A001  (tf.bool)
newaxis = None
Tensor = _torch.Tensor


def _t(x, dtype=None):
    """Anything -> torch tensor (numpy float64 stays float64 until cast, python floats become float32 like TF)."""
    if isinstance(x, _torch.Tensor):
        return x if dtype is None else x.to(dtype)
    if isinstance(x, _np.ndarray):
        t = _torch.from_numpy(_np.ascontiguousarray(x))
        return t if dtype is None else t.to(dtype)
    if isinstance(x, (list, tuple)) and len(x) and isinstance(x[0], _torch.Tensor):
        t = _torch.stack([_t(v) for v in x])
        return t if dtype is None else t.to(dtype)
    if dtype is None:
        if isinstance(x, float):
            dtype = _torch.float32
        elif isinstance(x, int) and not isinstance(x, _b.bool):
            dtype = _torch.int32
    return _torch.as_tensor(x, dtype=dtype)


def _i(x):
    """Shape entries / multiples may be python ints or 0-d tensors."""
    return int(x)


class Variable(_torch.nn.Parameter):
    """tf.Variable: a leaf tensor; trainable ones take part in GradientTape.gradient."""

    def __new__(cls, initial_value, trainable=True, dtype=None, name=None, **kwargs):
        t = _t(initial_value, dtype).detach().clone()
        trainable = _b.bool(trainable)
        return _torch.Tensor._make_subclass(cls, t, trainable and t.is_floating_point())

    def assign(self, value):
        with _torch.no_grad():
            self.copy_(_t(value).to(self.dtype))
        return self

    def numpy(self):
        return self.detach().numpy()

    def __deepcopy__(self, memo):
        return Variable(self.detach().clone(), trainable=self.requires_grad)


class TensorSpec:
    def __init__(self, shape=None, dtype=None, name=None):
        self.shape, self.dtype, self.name = shape, dtype, name


def function(func=None, input_signature=None, **kwargs):
    """tf.function: graph tracing has no numerical effect; the python function runs eagerly."""
    if func is not None:
        return func
    return lambda f: f


# ----------------------------------------------------------------------------------------------------------------------
# array ops
# ----------------------------------------------------------------------------------------------------------------------
def cast(x, dtype):
    return _t(x).to(dtype)


def convert_to_tensor(x, dtype=None):
    return _t(x, dtype)


def shape(x):
    return tuple(_t(x).shape)


def expand_dims(x, axis):
    return _t(x).unsqueeze(axis)


def squeeze(x, axis=None):
    x = _t(x)
    if axis is None:
        return x.squeeze()
    if isinstance(axis, (list, tuple)):
        return x.squeeze(tuple(axis))
    return x.squeeze(axis)


def reshape(x, shape):  # noqa: A002
    return _t(x).reshape([_i(s) for s in shape])


def transpose(x, perm=None):
    x = _t(x)
    if perm is None:
        perm = list(_b.range(x.dim()))[::-1]
    return x.permute(*[_i(p) for p in perm])


def concat(values, axis):
    return _torch.cat([_t(v) for v in values], dim=axis)


def tile(x, multiples):
    return _t(x).repeat(*[_i(m) for m in multiples])


def ones(shape, dtype=float32):  # noqa: A002
    if isinstance(shape, (int, _torch.Tensor)):
        shape = [shape]
    return _torch.ones([_i(s) for s in shape], dtype=dtype)


def zeros(shape, dtype=float32):  # noqa: A002
    if isinstance(shape, (int, _torch.Tensor)):
        shape = [shape]
    return _torch.zeros([_i(s) for s in shape], dtype=dtype)


def range(*args, dtype=None):  # noqa: A001
    return _torch.arange(*[_i(a) for a in args], dtype=dtype or _torch.int32)


def pad(x, paddings, constant_values=0):
    flat = []
    for lo, hi in reversed([list(p) for p in paddings]):
        flat += [_i(lo), _i(hi)]
    return _torch.nn.functional.pad(_t(x), flat, value=constant_values)


def _axis(axis):
    if isinstance(axis, list):
        return tuple(axis)
    return axis


def reduce_sum(x, axis=None, keepdims=False):
    x = _t(x)
    return x.sum() if axis is None else x.sum(dim=_axis(axis), keepdim=keepdims)


def reduce_mean(x, axis=None, keepdims=False):
    x = _t(x)
    return x.mean() if axis is None else x.mean(dim=_axis(axis), keepdim=keepdims)


def reduce_max(x, axis=None, keepdims=False):
    x = _t(x)
    return x.max() if axis is None else x.amax(dim=_axis(axis), keepdim=keepdims)


def argmax(x, axis=None):
    return _t(x).argmax(dim=axis)


def maximum(a, b):
    a, b = _t(a), _t(b)
    return _torch.maximum(a, b.to(a.dtype) if b.dtype != a.dtype else b)


def minimum(a, b):
    a, b = _t(a), _t(b)
    return _torch.minimum(a, b.to(a.dtype) if b.dtype != a.dtype else b)


def multiply(a, b):
    return _t(a) * _t(b)


def abs(x):  # noqa: A001
    return _t(x).abs()


def square(x):
    x = _t(x)
    return x * x


def matmul(a, b, transpose_a=False, transpose_b=False):
    a, b = _t(a), _t(b)
    if transpose_a:
        a = a.transpose(-1, -2)
    if transpose_b:
        b = b.transpose(-1, -2)
    return _torch.matmul(a, b)


math = _types.SimpleNamespace(
    equal=lambda a, b: _t(a) == (_t(b) if not isinstance(b, (int, float)) else b),
    logical_not=lambda a: ~_t(a),
    sqrt=lambda x: _t(x).sqrt(),
    round=lambda x: _torch.round(_t(x)),          # torch.round = round-half-to-even, as tf.math.round
    minimum=minimum, maximum=maximum, abs=abs,
    reduce_max=reduce_max, reduce_sum=reduce_sum, reduce_mean=reduce_mean, square=square,
)

nn = _types.SimpleNamespace(
    softmax=lambda x, axis=-1: _torch.softmax(_t(x), dim=axis),
    relu=lambda x: _torch.relu(_t(x)),
)


def _band_part(x, num_lower, num_upper):
    x = _t(x)
    out = x
    if num_lower >= 0:
        out = _torch.triu(out, diagonal=-num_lower)
    if num_upper >= 0:
        out = _torch.tril(out, diagonal=num_upper)
    return out


linalg = _types.SimpleNamespace(band_part=_band_part)


class TensorArray:
    def __init__(self, dtype, size=0, **kwargs):
        self._items = {}

    def write(self, index, value):
        self._items[_i(index)] = _t(value)
        return self

    def stack(self):
        return _torch.stack([self._items[k] for k in sorted(self._items)])


class RaggedTensor:
    """tf.RaggedTensor.from_row_lengths(values, row_lengths).to_tensor(): rows of `values` padded with zeros to the
    longest row."""

    def __init__(self, values, row_lengths):
        self.values = _t(values)
        self.row_lengths = [_i(v) for v in _t(row_lengths).reshape(-1).tolist()]
        if sum(self.row_lengths) != self.values.shape[0]:
            raise ValueError('row_lengths do not add up to the number of values')

    @classmethod
    def from_row_lengths(cls, values, row_lengths):
        return cls(values, row_lengths)

    def to_tensor(self):
        n = len(self.row_lengths)
        longest = max(self.row_lengths) if n else 0
        out = _torch.zeros((n, longest) + tuple(self.values.shape[1:]), dtype=self.values.dtype)
        pos = 0
        rows = []
        for r, ln in enumerate(self.row_lengths):
            rows.append(_torch.nn.functional.pad(self.values[pos:pos + ln], [0, 0] * (self.values.dim() - 1) + [0, longest - ln]))
            pos += ln
        return _torch.stack(rows) if rows else out


# ----------------------------------------------------------------------------------------------------------------------
# autograd
# ----------------------------------------------------------------------------------------------------------------------
class GradientTape:
    def __init__(self, persistent=False, watch_accessed_variables=True):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def gradient(self, target, sources):
        sources = list(sources)
        live = [s for s in sources if s.requires_grad]
        grads = _torch.autograd.grad(target, live, allow_unused=True, retain_graph=True)
        it = iter(grads)
        return [next(it) if s.requires_grad else None for s in sources]


# ----------------------------------------------------------------------------------------------------------------------
# Keras
# ----------------------------------------------------------------------------------------------------------------------
_name_counts = {}


def _auto_name(cls_name):
    n = _name_counts.get(cls_name, 0)
    _name_counts[cls_name] = n + 1
    snake = ''.join('_' + c.lower() if c.isupper() and i else c.lower() for i, c in enumerate(cls_name))
    return snake if n == 0 else f'{snake}_{n}'


class Layer:
    def __init__(self, name=None, trainable=True, dtype=None, **kwargs):
        self.name = name if name is not None else _auto_name(type(self).__name__)
        self.built = False

    def __call__(self, *args, **kwargs):
        return self.call(*args, **kwargs)

    def _children(self):
        for k, v in self.__dict__.items():
            if isinstance(v, (Layer, Variable)):
                yield k, v
            elif isinstance(v, (list, tuple)):
                for j, e in enumerate(v):
                    if isinstance(e, (Layer, Variable)):
                        yield f'{k}.{j}', e

    def named_variables(self, prefix=''):
        """Keras order (Layer.weights): the layer's OWN variables first, then its tracked sub-layers in the order they
        were assigned as attributes (lists flattened in place)."""
        return self._gather(prefix, True) + self._gather(prefix, False)

    def _gather(self, prefix, trainable):
        """Layer.weights = trainable_weights + non_trainable_weights, each: own variables, then the children's."""
        kids = list(self._children())
        out = [(prefix + k, v) for k, v in kids if isinstance(v, Variable) and v.requires_grad == trainable]
        for k, v in kids:
            if not isinstance(v, Variable):
                out.extend(v._gather(prefix + k + '.', trainable))
        return out

    @property
    def layers(self):
        return [v for _, v in self._children() if isinstance(v, Layer)]

    @property
    def variables(self):
        return [v for _, v in self.named_variables()]

    @property
    def trainable_variables(self):
        return [v for v in self.variables if v.requires_grad]


def _glorot_uniform(shape, fan_in, fan_out):
    lim = _math.sqrt(6.0 / (fan_in + fan_out))
    return (_torch.rand(shape) * 2 - 1) * lim


def _activation(name):
    if name is None or name == 'linear':
        return lambda x: x
    if name == 'relu':
        return _torch.relu
    raise NotImplementedError(f'activation {name!r} is not on the reference path')


class Dense(Layer):
    """keras.layers.Dense: activation(x @ kernel + bias); kernel (in, units) glorot_uniform, bias zeros."""

    def __init__(self, units, activation=None, use_bias=True, **kwargs):
        super().__init__(**kwargs)
        self.units = int(units)
        self._act = _activation(activation)
        self.kernel = None
        self.bias = None

    def call(self, x):
        x = _t(x)
        if not x.is_floating_point():
            x = x.float()
        if self.kernel is None:
            self.kernel = Variable(_glorot_uniform((x.shape[-1], self.units), x.shape[-1], self.units))
            self.bias = Variable(_torch.zeros(self.units))
        return self._act(_torch.matmul(x, self.kernel) + self.bias)


class Conv1D(Layer):
    """keras.layers.Conv1D, channels_last, stride 1: y[t] = sum_j x[t + j - pad_left] @ kernel[j] + bias; 'same' pads
    (k-1)//2 zeros on the left and k-1-(k-1)//2 on the right; kernel (k, in, filters)."""

    def __init__(self, filters, kernel_size, padding='valid', activation=None, **kwargs):
        super().__init__(**kwargs)
        self.filters, self.kernel_size, self.padding = int(filters), int(kernel_size), padding
        self._act = _activation(activation)
        self.kernel = None
        self.bias = None

    def call(self, x):
        x = _t(x)
        k = self.kernel_size
        if self.kernel is None:
            cin = x.shape[-1]
            self.kernel = Variable(_glorot_uniform((k, cin, self.filters), k * cin, k * self.filters))
            self.bias = Variable(_torch.zeros(self.filters))
        xt = x.transpose(1, 2)
        if self.padding == 'same':
            left = (k - 1) // 2
            xt = _torch.nn.functional.pad(xt, [left, k - 1 - left])
        elif self.padding != 'valid':
            raise NotImplementedError(self.padding)
        if xt.shape[-1] < k:
            y = _torch.zeros((x.shape[0], self.filters, 0), dtype=x.dtype)
        else:
            y = _torch.nn.functional.conv1d(xt, self.kernel.permute(2, 1, 0))
        return self._act(y.transpose(1, 2) + self.bias)


class LayerNormalization(Layer):
    """keras.layers.LayerNormalization(axis=-1): mean and BIASED variance over the last axis,
    (x - mean) * rsqrt(var + epsilon) * gamma + beta (the non-fused path Keras takes for epsilon < 1.001e-5)."""

    def __init__(self, axis=-1, epsilon=1e-3, **kwargs):
        super().__init__(**kwargs)
        self.epsilon = float(epsilon)
        self.gamma = None
        self.beta = None

    def call(self, x):
        x = _t(x)
        if self.gamma is None:
            self.gamma = Variable(_torch.ones(x.shape[-1]))
            self.beta = Variable(_torch.zeros(x.shape[-1]))
        mean = x.mean(dim=-1, keepdim=True)
        var = ((x - mean) ** 2).mean(dim=-1, keepdim=True)
        return (x - mean) * _torch.rsqrt(var + self.epsilon) * self.gamma + self.beta


class Embedding(Layer):
    def __init__(self, input_dim, output_dim, **kwargs):
        super().__init__(**kwargs)
        self.embeddings = Variable((_torch.rand(int(input_dim), int(output_dim)) * 2 - 1) * 0.05)

    def call(self, x):
        return self.embeddings[_t(x).long()]


class Dropout(Layer):
    """keras.layers.Dropout: identity unless training; kept values scaled by 1/(1-rate)."""

    def __init__(self, rate, **kwargs):
        super().__init__(**kwargs)
        object.__setattr__(self, 'rate', rate)

    def __setattr__(self, key, value):
        object.__setattr__(self, key, value)

    def _children(self):
        return iter(())  # `rate` may be a (non-trainable) Variable owned by the parent layer

    def call(self, x, training=False):
        rate = float(self.rate)
        if not training or rate <= 0.0:
            return x
        keep = (_torch.rand_like(x) >= rate).to(x.dtype)
        return x * keep / (1.0 - rate)


class Activation(Layer):
    def __init__(self, activation, **kwargs):
        super().__init__(**kwargs)
        self._act = _activation(activation)

    def call(self, x):
        return self._act(x)


class Model(Layer):
    def compile(self, optimizer=None, loss=None, loss_weights=None, **kwargs):
        self.optimizer = optimizer
        self.loss = loss
        self.compiled_loss_weights = loss_weights

    def save_weights(self, path):
        raise NotImplementedError('HDF5 export is not part of the shim')

    def load_weights(self, path):
        raise NotImplementedError('HDF5 import is not part of the shim')


class _Loss:
    def __init__(self, reduction='sum_over_batch_size', **kwargs):
        self.reduction = reduction

    def _reduce(self, per_sample, sample_weight):
        if sample_weight is not None:
            w = _t(sample_weight).to(per_sample.dtype)
            while w.dim() < per_sample.dim():
                w = w.unsqueeze(-1)
            per_sample = per_sample * w
        if self.reduction == 'none':
            return per_sample
        return per_sample.sum() / per_sample.numel()   # SUM_OVER_BATCH_SIZE divides by the number of elements


class MeanAbsoluteError(_Loss):
    def __call__(self, y_true, y_pred, sample_weight=None):
        y_pred = _t(y_pred)
        y_true = _t(y_true).to(y_pred.dtype)
        return self._reduce((y_pred - y_true).abs().mean(dim=-1), sample_weight)


class MeanSquaredError(_Loss):
    def __call__(self, y_true, y_pred, sample_weight=None):
        y_pred = _t(y_pred)
        y_true = _t(y_true).to(y_pred.dtype)
        return self._reduce(((y_pred - y_true) ** 2).mean(dim=-1), sample_weight)


class SparseCategoricalCrossentropy(_Loss):
    def __init__(self, from_logits=False, **kwargs):
        super().__init__(**kwargs)
        self.from_logits = from_logits

    def __call__(self, y_true, y_pred, sample_weight=None):
        y_pred = _t(y_pred)
        if not y_pred.is_floating_point():
            y_pred = y_pred.float()
        # float64 (numpy) logits: Keras computes in floatx = float32; evaluating in float64 and rounding the result once
        # reproduces the known answers of the reference's tests/test_loss.py to the last bit
        wide = y_pred.dtype == _torch.float64
        logp = _torch.log_softmax(y_pred, dim=-1) if self.from_logits else _torch.log(y_pred)
        idx = _t(y_true).long().unsqueeze(-1)
        out = self._reduce(-logp.gather(-1, idx).squeeze(-1), sample_weight)
        return out.float() if wide else out


class BinaryCrossentropy(_Loss):
    def __call__(self, y_true, y_pred, sample_weight=None):
        raise NotImplementedError('not on the reference path')


class Adam:
    """keras.optimizers.Adam (TF 2.2-2.4): lr_t = lr * sqrt(1 - b2^t) / (1 - b1^t); m, v EMA; theta -= lr_t * m / (sqrt(v) + eps)."""

    def __init__(self, learning_rate=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7, **kwargs):
        self.lr = Variable(float(learning_rate), trainable=False)
        self.beta_1, self.beta_2, self.epsilon = float(beta_1), float(beta_2), float(epsilon)
        self.iterations = Variable(_torch.zeros((), dtype=_torch.int64), trainable=False)
        self._slots = {}

    @property
    def learning_rate(self):
        return self.lr

    def apply_gradients(self, grads_and_vars):
        with _torch.no_grad():
            self.iterations.add_(1)
            t = int(self.iterations)
            lr_t = float(self.lr) * _math.sqrt(1.0 - self.beta_2 ** t) / (1.0 - self.beta_1 ** t)
            for g, v in grads_and_vars:
                if g is None:
                    continue
                m, s = self._slots.setdefault(id(v), (_torch.zeros_like(v), _torch.zeros_like(v)))
                m.mul_(self.beta_1).add_(g, alpha=1.0 - self.beta_1)
                s.mul_(self.beta_2).addcmul_(g, g, value=1.0 - self.beta_2)
                v.sub_(lr_t * m / (s.sqrt() + self.epsilon))


keras = _types.SimpleNamespace(
    layers=_types.SimpleNamespace(Layer=Layer, Dense=Dense, Conv1D=Conv1D, LayerNormalization=LayerNormalization,
                                  Embedding=Embedding, Dropout=Dropout, Activation=Activation),
    models=_types.SimpleNamespace(Model=Model),
    losses=_types.SimpleNamespace(MeanAbsoluteError=MeanAbsoluteError, MeanSquaredError=MeanSquaredError,
                                  SparseCategoricalCrossentropy=SparseCategoricalCrossentropy,
                                  BinaryCrossentropy=BinaryCrossentropy),
    optimizers=_types.SimpleNamespace(Adam=Adam),
)

random = _types.SimpleNamespace(set_seed=lambda s: _torch.manual_seed(int(s)))
config = _types.SimpleNamespace(experimental=_types.SimpleNamespace(list_physical_devices=lambda *_: [],
                                                                    set_memory_growth=lambda *_: None))
