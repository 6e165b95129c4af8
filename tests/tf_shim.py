"""TEST INFRASTRUCTURE ONLY: a minimal, FUNCTIONAL stand-in for the slice of TensorFlow 2.10 / Keras the
reference's hot path calls, built on PyTorch-CPU so that the reference's OWN graph code --
``create_model`` (scann/models/scann_model.py:329-453), ``LocalAttention.call`` / ``GlobalAttention.call`` /
``ResidualNorm.call`` (scann/layers/attention.py), ``GaussianExpansion.call`` / ``gather_shape`` / ``mrelu``
(scann/layers/custom_layers.py), ``root_mean_squared_error`` (scann/layers/losses.py) -- executes UNMODIFIED from
a checkout of the reference (SCANN_REFERENCE_ROOT), forward and (through torch autograd) backward.  TensorFlow itself is not installable here.

What this pins and what it does not.  Everything the reference *wrote* runs as written: which layers exist and in
which order, every einsum string, reshape, mask expression, concat order, residual, which Dense kernels carry
``regularizers.l2(1e-4)``, where Dropout sits, how ``ga_score`` is taken from ``global_attention``.  What comes from
this file instead of TensorFlow are the PRIMITIVES, restated from their documented semantics:

  Dense: ``x @ kernel + bias`` then activation ('swish' = x * sigmoid(x));  Embedding: row lookup;
  LayerNormalization(epsilon=1e-6): non-fused Keras path (eps < 1.001e-5) -- moments over the last axis (biased
  variance), ``tf.nn.batch_normalization``: inv = rsqrt(var + eps) * gamma, y = x * inv + (beta - mean * inv);
  Dropout: identity at inference, an injected pre-scaled keep mask in training;  softmax: max-subtracted;
  tf.linalg.normalize: x / sqrt(sum x^2) (0/0 = NaN as in TF);  regularizers.l2(c): c * sum(w^2);
  tf.gather_nd / einsum / concat / repeat / reshape / eye / reduce_sum / expand_dims: index arithmetic.

Functional-API calls run EAGERLY: ``Input(name=...)`` returns the fed tensor of that name, every layer call computes,
``tf.keras.Model(inputs, outputs)`` keeps the finished tensors.  Weights are not initialised here: a layer asks the
session for ``"<layer path>/<weight>"`` and gets the test's tensor (shape-checked), so the reference's weight inventory
is compared with ``scann_b200/params.py`` name by name.  Layer paths: top-level layers take their explicit ``name`` or
the Keras auto-name (snake-cased class name + per-class counter: ``local_attention``, ``local_attention_1`` ...);
a sub-layer takes its explicit ``name`` (``query``, ``key``, ``filter_geo``), else the attribute it is assigned to
(``layer_norm``, ``layer_norm_g``, ``drop_out``); members of a ``Sequential`` are auto-named per Sequential
(``dense``, ``dense_1``, ``dropout``) and the Sequential itself adds no path component.  (Real Keras auto-names
unnamed sub-layers with global counters; the names here are the ones ``scann_b200/params.py`` uses.)

Nothing under ``scann_b200/`` or ``scann/`` imports this module.
"""
from __future__ import annotations

import contextlib
import re
import sys
import types
from typing import Callable, Dict, List, Optional

import numpy as np
import torch


# ----------------------------------------------------------------------------------------------- session
class Session:
    """Everything one eager run of the reference graph needs: input feeds, weights, dropout masks."""

    def __init__(self, feeds: Dict[str, torch.Tensor], weights: Dict[str, torch.Tensor], dtype=torch.float64,
                 drop_masks: Optional[Dict[str, torch.Tensor]] = None):
        self.dtype = dtype
        self.feeds = feeds
        self.weights = weights
        self.drop_masks = drop_masks or {}
        self.counters: Dict[str, int] = {}
        self.top_layers: Dict[str, "Layer"] = {}
        self.used_weights: List[str] = []
        self.reg_losses: List[tuple] = []          # (weight name, penalty tensor)
        self.dropout_sites: List[str] = []         # paths of every Dropout that ran
        self.inputs_asked: List[str] = []

    def weight(self, name: str, shape) -> torch.Tensor:
        if name not in self.weights:
            raise KeyError(f"the reference graph asks for weight {name!r} {tuple(shape)}: not in the parameter layout")
        w = self.weights[name]
        if tuple(w.shape) != tuple(int(s) for s in shape):
            raise ValueError(f"weight {name}: reference shape {tuple(shape)} != layout shape {tuple(w.shape)}")
        if name not in self.used_weights:
            self.used_weights.append(name)
        return w

    def auto_name(self, cls_name: str) -> str:
        base = _snake(cls_name)
        i = self.counters.get(base, 0)
        self.counters[base] = i + 1
        return base if i == 0 else f"{base}_{i}"


_session: Optional[Session] = None


@contextlib.contextmanager
def session(feeds, weights, dtype=torch.float64, drop_masks=None):
    """Runs the body with a fresh Session; the shim's module tree is importable as ``tensorflow`` meanwhile
    (``gather_shape`` does ``import tensorflow as tf`` at call time, custom_layers.py:19)."""
    global _session
    prev, _session = _session, Session(feeds, weights, dtype, drop_masks)
    saved = {k: v for k, v in sys.modules.items() if k == "tensorflow" or k.startswith("tensorflow.")}
    for k in saved:
        del sys.modules[k]
    sys.modules.update(build_modules())
    try:
        yield _session
    finally:
        _session = prev
        for k in [k for k in sys.modules if k == "tensorflow" or k.startswith("tensorflow.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def _S() -> Session:
    if _session is None:
        raise RuntimeError("tf_shim: no session (use `with tf_shim.session(feeds, weights): ...`)")
    return _session


def _snake(name: str) -> str:
    s = re.sub(r"(.)([A-Z][a-z0-9]+)", r"\1_\2", name)
    return re.sub(r"([a-z])([A-Z])", r"\1_\2", s).lower()


class DType:
    def __init__(self, name, floating):
        self.name, self.floating = name, floating

    def __repr__(self):
        return f"tf.{self.name}"


float32 = DType("float32", True)     # maps to the session's working dtype (fp64 for truth, fp32 for the reference's rounding)
float64 = DType("float64", True)
int32 = DType("int32", False)
int64 = DType("int64", False)
bool_ = DType("bool", False)


def _torch_dtype(d):
    if isinstance(d, DType):
        d = d.name
    if isinstance(d, torch.dtype):
        return d
    d = str(d)
    if d in ("float32", "float64", "float"):
        return _S().dtype
    if d in ("int32", "int64", "int"):
        return torch.int64
    if d == "bool":
        return torch.bool
    raise TypeError(d)


def _t(x):
    """tf.convert_to_tensor: numpy float arrays / python floats take the working dtype."""
    if isinstance(x, torch.Tensor):
        return x
    a = np.asarray(x)
    if a.dtype.kind == "f":
        return torch.as_tensor(a.astype(np.float64)).to(_S().dtype)
    if a.dtype.kind in "iu":
        return torch.as_tensor(a.astype(np.int64))
    if a.dtype.kind == "b":
        return torch.as_tensor(a)
    raise TypeError(a.dtype)


# ----------------------------------------------------------------------------------------------- tf.*
def shape(x):
    return [int(s) for s in _t(x).shape]


def cast(x, dtype):
    td = _torch_dtype(dtype)
    if isinstance(x, (int, float)) and not isinstance(x, bool):
        return float(x) if td.is_floating_point else int(x)
    return _t(x).to(td)


def reshape(x, shp):
    return _t(x).reshape([int(s) for s in shp])


def concat(values, axis):
    vals = [_t(v) for v in values]
    if any(v.dtype.is_floating_point for v in vals):
        vals = [v.to(_S().dtype) for v in vals]
    return torch.cat(vals, int(axis))


def repeat(x, repeats, axis=None):
    return torch.repeat_interleave(_t(x), int(repeats), dim=axis)


def expand_dims(x, axis):
    return _t(x).unsqueeze(int(axis))


def gather_nd(params, indices):
    idx = _t(indices).long()
    return _t(params)[tuple(idx[..., k] for k in range(idx.shape[-1]))]


def multiply(a, b):
    return _t(a) * (b if isinstance(b, (int, float)) else _t(b))


def maximum(a, b):
    a = _t(a)
    return torch.maximum(a, torch.as_tensor(b, dtype=a.dtype) if isinstance(b, (int, float)) else _t(b))


def einsum(eq, *ops):
    return torch.einsum(eq.replace(" ", ""), *[_t(o) for o in ops])


def reduce_sum(x, axis=None):
    x = _t(x)
    return x.sum() if axis is None else x.sum(int(axis))


def eye(n, batch_shape=None, dtype="float32"):
    e = torch.eye(int(n), dtype=_torch_dtype(dtype))
    if batch_shape is not None:
        e = e.expand(*[int(b) for b in batch_shape], int(n), int(n))
    return e


def range_(n):
    return torch.arange(int(n), dtype=torch.int64)


def broadcast_to(x, shp):
    return _t(x).expand(*[int(s) for s in shp])


def ones(shp, dtype="float32"):
    return torch.ones(*[int(s) for s in shp], dtype=_torch_dtype(dtype))


def Variable(initial_value, dtype=None, name=None, **kw):
    return _t(initial_value)


def custom_gradient(f: Callable):
    """@tf.custom_gradient: f(x) -> (y, grad_fn); the backward pass calls grad_fn(dy)."""

    class _Fn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x):
            with torch.enable_grad():
                y, grad_fn = f(x.detach())
            ctx.grad_fn_ = grad_fn
            return y.detach()

        @staticmethod
        def backward(ctx, dy):
            return ctx.grad_fn_(dy)

    def wrapped(x):
        return _Fn.apply(_t(x))

    wrapped.__name__ = getattr(f, "__name__", "custom_gradient")
    return wrapped


def _exp(x):
    return torch.exp(_t(x))


def _logical_not(x):
    return torch.logical_not(_t(x))


def _softmax(x, axis=-1):
    return torch.softmax(_t(x), int(axis))


def _normalize(tensor, ord="euclidean", axis=None, name=None):
    assert ord == "euclidean"
    x = _t(tensor)
    norm = torch.sqrt((x * x).sum(int(axis), keepdim=True))
    return x / norm, norm


# ----------------------------------------------------------------------------------------------- keras layers
class Layer:
    def __init__(self, name=None, dtype=None, trainable=True, **kwargs):
        d = self.__dict__
        d["_explicit_name"] = name
        d.setdefault("_parent", None)
        d.setdefault("_attr", None)
        d["_path_cache"] = None
        d["output"] = None

    def __setattr__(self, key, value):
        if isinstance(value, Layer) and not key.startswith("_") and value.__dict__.get("_parent") is None:
            value.__dict__["_parent"] = self
            value.__dict__["_attr"] = key
            self.__dict__.setdefault("_tracked", []).append(value)      # Keras tracks sub-layers in assignment order
        object.__setattr__(self, key, value)

    OWN_WEIGHTS: tuple = ()

    def weights_order(self) -> List[str]:
        """Names (full paths) of ``layer.weights`` in Keras order: the layer's own variables, then those of its
        tracked sub-layers in attribute-assignment order -- the order of ``weight_names`` in a Keras HDF5 file."""
        p = self.path()
        out = [f"{p}/{w}" for w in self.OWN_WEIGHTS]
        for sub in self.__dict__.get("_tracked", []):
            out += sub.weights_order()
        return out

    # -- naming
    def _own_name(self) -> str:
        d = self.__dict__
        return d.get("_explicit_name") or d.get("_seq_name") or d.get("_attr")

    def path(self) -> str:
        d = self.__dict__
        if d.get("_path_cache") is None:
            parent = d.get("_parent")
            if parent is None:
                name = d.get("_explicit_name") or _S().auto_name(type(self).__name__)
                _S().top_layers[name] = self
                d["_path_cache"] = name
            else:
                pp = parent.path()
                own = self._own_name()
                d["_path_cache"] = own if pp == "" else f"{pp}/{own}"
        return d["_path_cache"]

    @property
    def name(self):
        return self.path().split("/")[-1]

    def __call__(self, *args, **kwargs):
        self.path()                                   # fixes the auto-name in call order
        out = self.call(*args, **kwargs)
        self.__dict__["output"] = list(out) if isinstance(out, tuple) else out
        return out

    def call(self, *args, **kwargs):
        raise NotImplementedError

    def get_config(self):
        return {"name": self.name}


def _activation(act):
    if act is None or act == "linear":
        return lambda y: y
    if act == "swish":
        return lambda y: y * torch.sigmoid(y)
    if callable(act):
        return act
    raise NotImplementedError(f"activation {act!r}")


class Dense(Layer):
    OWN_WEIGHTS = ("kernel", "bias")

    def get_config(self):
        act = self.activation
        return {"name": self.name, "units": self.units,
                "activation": "linear" if act is None else act if isinstance(act, str) else getattr(act, "__name__", "?")}

    def __init__(self, units, activation=None, kernel_regularizer=None, **kwargs):
        super().__init__(**kwargs)
        self.units = int(units)
        self.activation = activation
        self.kernel_regularizer = kernel_regularizer

    def call(self, x):
        x = _t(x).to(_S().dtype)                      # Dense.call casts its input to the compute dtype
        p = self.path()
        k = _S().weight(f"{p}/kernel", (x.shape[-1], self.units))
        b = _S().weight(f"{p}/bias", (self.units,))
        if self.kernel_regularizer is not None and all(n != f"{p}/kernel" for n, _ in _S().reg_losses):
            _S().reg_losses.append((f"{p}/kernel", self.kernel_regularizer(k)))
        return _activation(self.activation)(x @ k + b)


class Embedding(Layer):
    OWN_WEIGHTS = ("embeddings",)

    def get_config(self):
        return {"name": self.name, "input_dim": self.input_dim, "output_dim": self.output_dim}

    def __init__(self, input_dim, output_dim, **kwargs):
        super().__init__(**kwargs)
        self.input_dim, self.output_dim = int(input_dim), int(output_dim)

    def call(self, x):
        return _S().weight(f"{self.path()}/embeddings", (self.input_dim, self.output_dim))[_t(x).long()]


class Dropout(Layer):
    """Inference: identity.  Training: multiplies by the injected mask of this site (0 or 1/keep, as Keras)."""

    def __init__(self, rate, **kwargs):
        super().__init__(**kwargs)
        self.rate = float(rate)

    def get_config(self):
        return {"name": self.name, "rate": self.rate}

    def call(self, x):
        p = self.path()
        _S().dropout_sites.append(p)
        m = _S().drop_masks.get(p)
        return x if m is None else x * _t(m).reshape(x.shape)


class LayerNormalization(Layer):
    OWN_WEIGHTS = ("gamma", "beta")

    def __init__(self, epsilon=1e-3, **kwargs):
        super().__init__(**kwargs)
        self.epsilon = float(epsilon)
        assert self.epsilon < 1.001e-5, "only the non-fused Keras path is restated"

    def call(self, x):
        p = self.path()
        gamma = _S().weight(f"{p}/gamma", (x.shape[-1],))
        beta = _S().weight(f"{p}/beta", (x.shape[-1],))
        mean = x.mean(-1, keepdim=True)
        var = ((x - mean) ** 2).mean(-1, keepdim=True)
        inv = torch.rsqrt(var + self.epsilon) * gamma
        return x * inv + (beta - mean * inv)


class Add(Layer):
    def call(self, xs):
        out = _t(xs[0])
        for v in xs[1:]:
            out = out + _t(v)
        return out


class Multiply(Layer):
    def call(self, xs):
        out = _t(xs[0])
        for v in xs[1:]:
            out = out * _t(v)
        return out


class Lambda(Layer):
    def __init__(self, function, **kwargs):
        super().__init__(**kwargs)
        self.function = function

    def call(self, x):
        return self.function(x)


class Sequential(Layer):
    """Transparent for naming: its members hang under the Sequential's owner."""

    def __init__(self, layers=None, **kwargs):
        super().__init__(**kwargs)
        counters: Dict[str, int] = {}
        self._layers = list(layers or [])
        for l in self._layers:
            base = _snake(type(l).__name__)
            i = counters.get(base, 0)
            counters[base] = i + 1
            l.__dict__["_parent"] = self
            l.__dict__["_seq_name"] = base if i == 0 else f"{base}_{i}"
            self.__dict__.setdefault("_tracked", []).append(l)

    def path(self) -> str:
        parent = self.__dict__.get("_parent")
        return "" if parent is None else parent.path()

    def call(self, x):
        for l in self._layers:
            x = l(x)
        return x


def Input(shape=None, name=None, dtype="float32", **kwargs):
    s = _S()
    if name not in s.feeds:
        raise KeyError(f"the reference graph declares Input {name!r}: not fed")
    s.inputs_asked.append(name)
    return _t(s.feeds[name]).to(_torch_dtype(dtype))


class Model:
    def __init__(self, inputs=None, outputs=None, **kwargs):
        self.inputs = list(inputs) if isinstance(inputs, (list, tuple)) else [inputs]
        self.outputs = list(outputs) if isinstance(outputs, (list, tuple)) else [outputs]
        self.input, self.output = inputs, outputs
        self._session = _S()

    def summary(self, *a, **k):
        pass

    def get_layer(self, name):
        return self._session.top_layers[name]

    @property
    def losses(self):
        return [t for _, t in self._session.reg_losses]


class L2:
    def __init__(self, l2=0.01):
        self.l2 = float(l2)

    def __call__(self, w):
        return self.l2 * (w * w).sum()


class Callback:
    """Base of the reference's own callbacks (SGDRC, LearningRateLoggingCallback) and of the RECORDING stand-ins for
    the stock Keras callbacks / optimisers below: those keep their constructor arguments for the shell-level tests
    (what the reference's ``create_callbacks`` / ``train`` asks Keras for); none of them trains anything."""

    def __init__(self, *args, **kwargs):
        self.model = None
        self.args, self.kwargs = args, kwargs


def _recording(name):
    return type(name, (Callback,), {})


class _Recorder:
    def __init__(self, *args, **kwargs):
        self.args, self.kwargs = args, kwargs


# ----------------------------------------------------------------------------------------------- module tree
def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__path__ = []                                   # a package: inert stubs may serve submodules it lacks
    m.__dict__.update(attrs)
    return m


_modules: Optional[Dict[str, types.ModuleType]] = None


def build_modules() -> Dict[str, types.ModuleType]:
    """-> {"tensorflow": ..., "tensorflow.keras": ..., ...} ready for sys.modules (one tree per process)."""
    global _modules
    if _modules is not None:
        return _modules
    backend = _mod("tensorflow.keras.backend", sqrt=lambda x: torch.sqrt(_t(x)), mean=lambda x, axis=None: _t(x).mean()
                   if axis is None else _t(x).mean(axis), square=lambda x: _t(x) ** 2,
                   sum=lambda x, axis=None: reduce_sum(x, axis), epsilon=lambda: 1e-7)
    regularizers = _mod("tensorflow.keras.regularizers", l2=L2, L2=L2)
    callbacks = _mod("tensorflow.keras.callbacks", Callback=Callback, ModelCheckpoint=_recording("ModelCheckpoint"),
                     EarlyStopping=_recording("EarlyStopping"), CSVLogger=_recording("CSVLogger"),
                     ReduceLROnPlateau=_recording("ReduceLROnPlateau"),
                     LearningRateScheduler=_recording("LearningRateScheduler"))
    schedules = _mod("tensorflow.keras.optimizers.schedules", CosineDecay=type("CosineDecay", (_Recorder,), {}))
    optimizers = _mod("tensorflow.keras.optimizers", Adam=type("Adam", (_Recorder,), {}), schedules=schedules)
    backend_extra = dict(clear_session=lambda: None)
    layers = _mod("tensorflow.keras.layers", Layer=Layer, Dense=Dense, Dropout=Dropout, Embedding=Embedding, Input=Input,
                  Lambda=Lambda, Multiply=Multiply, Add=Add, LayerNormalization=LayerNormalization)

    def load_model(*a, **k):
        raise NotImplementedError("tf_shim: load_model (Keras HDF5) is outside the shim; see scann_b200/h5lite.py")

    models = _mod("tensorflow.keras.models", load_model=load_model, Model=Model, Sequential=Sequential)
    backend.__dict__.update(backend_extra)
    keras = _mod("tensorflow.keras", backend=backend, regularizers=regularizers, callbacks=callbacks, layers=layers,
                 models=models, optimizers=optimizers, Model=Model, Sequential=Sequential, Input=Input)
    math = _mod("tensorflow.math", exp=_exp, logical_not=_logical_not)
    nn = _mod("tensorflow.nn", softmax=_softmax)
    linalg = _mod("tensorflow.linalg", normalize=_normalize)
    tf = _mod("tensorflow", keras=keras, math=math, nn=nn, linalg=linalg, shape=shape, cast=cast, reshape=reshape,
              concat=concat, repeat=repeat, expand_dims=expand_dims, gather_nd=gather_nd, multiply=multiply,
              maximum=maximum, einsum=einsum, reduce_sum=reduce_sum, eye=eye, range=range_, broadcast_to=broadcast_to,
              ones=ones, Variable=Variable, custom_gradient=custom_gradient, float32=float32, float64=float64,
              int32=int32, int64=int64, bool=bool_, __version__="2.10.0-shim")
    _modules = {m.__name__: m for m in (tf, keras, backend, regularizers, callbacks, layers, models, optimizers, schedules, math, nn,
                                       linalg)}
    return _modules
