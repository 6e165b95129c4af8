"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  Not part of the product path.

Op-for-op restatement, in PyTorch-CPU, of the reference's TensorFlow/Keras graph for the
SCANN attention hot path.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import this module.

PARITY: PINNED TO REFERENCE-RUN CODE AT THE GRAPH LEVEL, UNPINNED AT THE TENSORFLOW-PRIMITIVE LEVEL.
The reference's arithmetic lives in TensorFlow 2.10 / Keras 2.10 (environment.yml:144,212,282), which is neither
installed nor installable here (no wheel, no network), and the reference ships no tests, golden vectors or weights
(SURVEY.md F2, F8).  What IS checked (tests/test_reference_graph.py, run where SCANN_REFERENCE_ROOT
names a checkout of the reference): the reference's own ``create_model`` / ``LocalAttention.call`` / ``GlobalAttention.call`` /
``ResidualNorm.call`` / ``GaussianExpansion`` / ``gather_shape`` / ``mrelu`` / ``root_mean_squared_error`` are imported
UNMODIFIED and executed on a functional stand-in for the TensorFlow primitives (tests/tf_shim.py, PyTorch-CPU); this
restatement agrees with them to fp64 round-off on outputs, ga_score, loss and every per-tensor gradient for seven
configurations (SCANN+ / SCANN, ring, cgcnn, mrelu head, with / without ResidualNorm and ga normalisation, injected
Dropout masks, no-neighbour atoms, single-atom NaN), and the golden vectors in ``tests/golden`` equal that run.
What is NOT checked: TensorFlow's own kernels behind those primitives (fp32 summation order of its GEMMs /
reductions, fused vs non-fused LayerNormalization) -- restated from the Keras documentation: non-fused
LayerNormalization for eps < 1.001e-5, max-subtracted softmax, swish = x*sigmoid(x), Dense = x @ W + b.

Every function cites the reference lines it follows (paths relative to the reference's repository root).
Run in float64 for "truth" and in float32 for the reference's own rounding behaviour.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

L2_COEF = 1e-4     # regularizers.l2(1e-4)  (attention.py:27-28,95,97,108,260,262; scann_model.py:428,441)
LN_EPS = 1e-6      # LayerNormalization(epsilon=1e-6) (attention.py:35,111,113)
N_RBF = 20


# --------------------------------------------------------------------------- primitives
def swish(x: torch.Tensor) -> torch.Tensor:
    """keras 'swish' activation: x * sigmoid(x)."""
    return x * torch.sigmoid(x)


def layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor) -> torch.Tensor:
    """Keras LayerNormalization, non-fused path (eps=1e-6 < 1.001e-5 disables the fused
    kernel): biased variance from tf.nn.moments, then tf.nn.batch_normalization:
    inv = rsqrt(var + eps) * gamma ; y = x * inv + (beta - mean * inv)."""
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    inv = torch.rsqrt(var + LN_EPS) * gamma
    return x * inv + (beta - mean * inv)


def dense(x: torch.Tensor, w: Dict[str, torch.Tensor], name: str, act=None) -> torch.Tensor:
    """keras Dense on rank>=2 input: x @ kernel + bias."""
    y = x @ w[f"{name}/kernel"] + w[f"{name}/bias"]
    return act(y) if act is not None else y


class _MRelu(torch.autograd.Function):
    """mrelu: max(x,0) forward, identity gradient (scann/layers/custom_layers.py:6-15)."""

    @staticmethod
    def forward(ctx, x):
        return torch.clamp_min(x, 0.0)

    @staticmethod
    def backward(ctx, dy):
        return dy


def mrelu(x: torch.Tensor) -> torch.Tensor:
    return _MRelu.apply(x)


def rbf_centers(hi: float) -> np.ndarray:
    """np.linspace(0, hi, 20, dtype='float32') (scann_model.py:378, :384)."""
    return np.linspace(0, hi, N_RBF, dtype="float32")


def gaussian_expansion(d: torch.Tensor, centers: np.ndarray, width: float = 0.5) -> torch.Tensor:
    """GaussianExpansion.call (custom_layers.py:55-65); the ctor stores width**2 (:48-51)."""
    c = torch.as_tensor(centers).to(d.dtype)          # fp32 constants, widened for the fp64 run
    return torch.exp(-((d.unsqueeze(-1) - c) ** 2) / (width ** 2))


def gather_shape(neighbors: torch.Tensor) -> torch.Tensor:
    """gather_shape (custom_layers.py:18-28): [B,M,N] -> [B,M,N,2] = (batch id, neighbour id)."""
    B, M, N = neighbors.shape
    rb = torch.arange(B, dtype=neighbors.dtype).view(B, 1, 1, 1).expand(B, M, N, 1)
    return torch.cat([rb, neighbors.unsqueeze(-1)], -1)


def gather_nd(x: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """tf.gather_nd(atom_query, atom_neighbor) (attention.py:136): x[B,M,D], idx[B,M,N,2]."""
    return x[idx[..., 0].long(), idx[..., 1].long()]


# --------------------------------------------------------------------------- layers
def local_attention(w, name, x, idx, geom, mask, weight=None, *, g_update: bool, num_head: int = 8,
                    scale: float = 0.5, attn_drop_mask: Optional[torch.Tensor] = None):
    """LocalAttention.call with v_proj=False, kq_proj=True (attention.py:118-216).

    x[B,M,D]; idx[B,M,N,2]; geom [B,M,N,D] (g_update) or [B,M,N,20]; mask[B,M,N] float;
    weight [B,M,N,1] (g_update=False).  Returns (attn[B,H,M,N], context[B,M,D], geom'[B,M,N,D]).
    ``attn_drop_mask`` (already scaled by 1/keep) stands in for Dropout(0.05) (:191-192).
    """
    B, M, N = idx.shape[:3]
    D = x.shape[-1]
    hd = D // num_head
    nbr = gather_nd(x, idx).reshape(B, M, N, D)                                        # :136-139
    if g_update:
        cat = torch.cat([x.unsqueeze(2).expand(B, M, N, D), geom, nbr], -1)            # :143-150
        upd = dense(cat, w, f"{name}/filter_geo", swish)                               # :142
        geom = layer_norm(upd + geom, w[f"{name}/layer_norm_g/gamma"], w[f"{name}/layer_norm_g/beta"])  # :153
    else:
        geom = dense(geom, w, f"{name}/filter_geo", swish) * weight                    # :155
    a = nbr * geom                                                                     # :157
    q = dense(x, w, f"{name}/query")                                                   # :160
    k = dense(a, w, f"{name}/key")                                                     # :163
    qt = q.reshape(B, M, num_head, hd)                                                 # :170
    kt = k.reshape(B, M, N, num_head, hd)                                              # :173
    dk = float(hd) ** (-scale)                                                         # :180
    qt = qt * dk                                                                       # :181
    energy = torch.einsum("bchd,bcnhd->bhcn", qt, kt)                                  # :183
    energy = energy + (1.0 - mask.unsqueeze(1)) * -1e9                                 # :186-187
    attn = torch.softmax(energy, -1)                                                   # :189
    if attn_drop_mask is not None:
        attn = attn * attn_drop_mask                                                   # :191-192
    ctx = torch.einsum("bcn,bcnhd->bcnhd", mask, torch.einsum("bhcn,bcnhd->bcnhd", attn, kt))  # :206
    ctx = ctx.reshape(B, M, N, D)                                                      # :208
    ctx = ctx.sum(2) + q                                                               # :212 (q unscaled)
    ctx = layer_norm(ctx, w[f"{name}/layer_norm/gamma"], w[f"{name}/layer_norm/beta"])  # :214
    return attn, ctx, geom


def residual_norm(w, name, x, drop_mask: Optional[torch.Tensor] = None):
    """ResidualNorm.call (attention.py:37-40; Sequential :25-31)."""
    h = dense(x, w, f"{name}/dense", swish)
    h = dense(h, w, f"{name}/dense_1")
    if drop_mask is not None:
        h = h * drop_mask
    return layer_norm(x + h, w[f"{name}/layer_norm/gamma"], w[f"{name}/layer_norm/beta"])


def global_attention(w, name, x, mask, *, norm: bool):
    """GlobalAttention.call with v_proj=False, kq_proj=True (attention.py:267-318).
    x[B,M,D], mask[B,M,1] -> (attn[B,M,1] = ga_score, context[B,D])."""
    B, M, _ = x.shape
    q = dense(x, w, f"{name}/query")                                                   # :269
    k = dense(x, w, f"{name}/key")                                                     # :272
    energy = torch.einsum("bkd,bqd->bkq", mask * k, mask * q)                          # :279
    not_eye = 1.0 - torch.eye(M, dtype=x.dtype).unsqueeze(0)                           # :282-283
    energy = not_eye * energy                                                          # :285
    agg = energy.sum(-1).reshape(B, -1, 1)                                             # :289-290
    agg = mask * agg                                                                   # :292
    if norm:
        # tf.linalg.normalize(ord='euclidean', axis=1): x / sqrt(sum(x^2)), no epsilon   :297
        agg = agg / torch.sqrt((agg * agg).sum(1, keepdim=True))
    agg = agg + (1.0 - mask) * -1e9                                                    # :299-300
    attn = torch.softmax(agg, 1)                                                       # :302
    ctx = (mask * (attn * k)).sum(1)                                                   # :314-316
    return attn, ctx


def _name(base: str, i: int) -> str:
    return base if i == 0 else f"{base}_{i}"


# --------------------------------------------------------------------------- whole graph
def forward(w: Dict[str, torch.Tensor], inputs: Dict[str, torch.Tensor], *, n_attention: int,
            g_update: bool, gaussian_d: float, use_attn_norm: bool, use_ga_norm: bool,
            use_ring: bool = False, num_head: int = 8, mrelu_head: bool = False,
            drop_masks: Optional[Dict[str, torch.Tensor]] = None, return_all: bool = False):
    """create_model (scann_model.py:329-453), 'atomic' feature.  Returns (y[B,1], ga[B,M,1]).

    ``inputs`` follow the reference's Input layers (:338-358); masks are float tensors
    (Keras casts the bool arrays to float32).  ``drop_masks`` optionally injects the
    training-mode dropout masks (pre-scaled by 1/keep): keys 'dense_embed',
    'residual_norm_<l>', 'local_attention_<l>'.
    """
    dm = drop_masks or {}
    dtype = inputs["neighbor_distance"].dtype
    atom_mask = inputs["atom_mask"].to(dtype)
    nmask = inputs["neighbor_mask"].to(dtype)
    if "embed_atom/kernel" in w:                       # feature == "cgcnn": [B,M,92] features, Dense embedding
        x = dense(inputs["atomic"].to(dtype), w, "embed_atom")                         # :364-365
    else:
        x = w["embed_atom/embeddings"][inputs["atomic"].long()]                        # :362
    if use_ring:
        ring = dense(inputs["ring_aromatic"].to(dtype), w, "extra_embed")              # :368
        x = torch.cat([x, ring], -1)                                                   # :371
    x = dense(x, w, "dense_embed", swish)                                              # :373
    if "dense_embed" in dm:
        x = x * dm["dense_embed"]                                                      # :374
    idx = gather_shape(inputs["neighbors"].long())                                     # :376
    rbf = gaussian_expansion(inputs["neighbor_distance"], rbf_centers(gaussian_d))     # :378
    if g_update:
        gd = dense(rbf, w, "neighbor_d", swish)                                        # :381
        gw = gaussian_expansion(inputs["neighbor_weight"], rbf_centers(np.pi * 2))     # :384
        gw = dense(gw, w, "neighbor_w", swish)                                         # :386
        geom = gd * gw                                                                 # :389
        nw = None
    else:
        geom = rbf
        nw = inputs["neighbor_weight"].unsqueeze(-1)                                   # :391
    trace = {"x0": x, "g0": geom}
    for l in range(n_attention):                                                       # :413-421
        la = _name("local_attention", l)
        attn, ctx, g_new = local_attention(w, la, x, idx, geom, nmask, nw, g_update=g_update,
                                           num_head=num_head, attn_drop_mask=dm.get(la))
        x = residual_norm(w, _name("residual_norm", l), ctx, dm.get(_name("residual_norm", l))) \
            if use_attn_norm else ctx                                                  # :404-408
        if g_update:
            geom = g_new                                                               # :415-417
        trace[f"attn{l}"] = attn
        trace[f"ctx{l}"] = ctx
        trace[f"x{l + 1}"] = x
        trace[f"g{l + 1}"] = g_new
    x = dense(x, w, "after_Lc", swish)                                                 # :424-429
    ga, s = global_attention(w, "global_attention", x, atom_mask, norm=use_ga_norm)    # :432-434
    s = dense(s, w, "bf_property", swish)                                              # :437-442
    y = dense(s, w, "predict_property", mrelu if mrelu_head else None)                 # :445-447
    if return_all:
        trace["after_Lc"] = x
        return y, ga, trace
    return y, ga


def l2_penalty(w: Dict[str, torch.Tensor], l2_names) -> torch.Tensor:
    """Sum of kernel_regularizer terms Keras adds to the loss: 1e-4 * sum(W^2)."""
    return sum(L2_COEF * (w[n] ** 2).sum() for n in l2_names)


def rmse_loss(y_true: torch.Tensor, y_pred: torch.Tensor) -> torch.Tensor:
    """root_mean_squared_error (scann/layers/losses.py:5-6); Keras aligns y_true[B] -> [B,1]."""
    return torch.sqrt(torch.mean((y_pred - y_true.reshape(-1, 1)) ** 2))


def loss_and_grads(w_np: Dict[str, np.ndarray], inputs_np: Dict[str, np.ndarray], target: np.ndarray,
                   l2_names, dtype=torch.float64, **model_kw):
    """One Keras train_step's loss and gradients (scann_model.py:210-241): RMSE + l2 terms,
    reverse-mode autodiff.  Returns (loss, y, ga, grads dict)."""
    w = {k: torch.tensor(np.asarray(v), dtype=dtype, requires_grad=True) for k, v in w_np.items()}
    inputs = to_torch_inputs(inputs_np, dtype)
    y, ga = forward(w, inputs, **model_kw)
    loss = rmse_loss(torch.tensor(target, dtype=dtype), y) + l2_penalty(w, l2_names)
    loss.backward()
    grads = {k: (v.grad.numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in w.items()}
    return float(loss.detach()), y.detach().numpy(), ga.detach().numpy(), grads


def to_torch_inputs(inputs_np: Dict[str, np.ndarray], dtype=torch.float64) -> Dict[str, torch.Tensor]:
    out = {}
    for k, v in inputs_np.items():
        v = np.asarray(v)
        if k == "neighbors" or (k == "atomic" and v.ndim == 2):
            out[k] = torch.tensor(v.astype(np.int64))
        else:
            out[k] = torch.tensor(v.astype(np.float64)).to(dtype)
    return out


def predict(w_np: Dict[str, np.ndarray], inputs_np: Dict[str, np.ndarray], dtype=torch.float64, **model_kw):
    """SCANN(..., mode='infer').model.predict(inputs) -> (target[B,1], ga_score[B,M,1])
    (scann_model.py:79-83)."""
    with torch.no_grad():
        w = {k: torch.tensor(np.asarray(v), dtype=dtype) for k, v in w_np.items()}
        y, ga = forward(w, to_torch_inputs(inputs_np, dtype), **model_kw)
    return y.numpy(), ga.numpy()


# --------------------------------------------------------------------------- optimiser (train step)
def adam_legacy_step(p, g, m, v, step: int, lr: float, decay: float = 1e-5, b1=0.9, b2=0.999, eps=1e-7):
    """tf.keras.optimizers.Adam(lr, decay=1e-5) of Keras 2.10 (scann_model.py:212): OptimizerV2
    with the legacy ``decay`` hyper-parameter, lr_t = lr / (1 + decay*iterations) where
    ``iterations`` is the count BEFORE this update, then the standard bias-corrected update
    with epsilon=1e-7 outside the sqrt.  ``step`` is 1-based."""
    lr_t = lr / (1.0 + decay * (step - 1))
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    alpha = lr_t * np.sqrt(1 - b2 ** step) / (1 - b1 ** step)
    p = p - alpha * m / (np.sqrt(v) + eps)
    return p, m, v
