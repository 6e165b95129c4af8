"""The train step's kernel families, one launch at a time, against plain fp64 restatements (torch float64 on the CPU).

* ``scann_wgrad_batch_tc``, ``scann_wgrad_batch_tc_det`` + ``scann_wgrad_batch_reduce``: every dW += X^T Y and
  db += colsum(Y) of a step in one launch -- pair problems on real pair plans (tile slots of 32, 64 and 128 rows, atoms
  with more than 32 neighbours), with and without the compact list of valid rows; per-atom problems with ragged row
  counts and strided operands; grids that split one problem between CTAs or pack many problems into one CTA; the
  longest table one launch takes.
* ``scann_dense_chain2`` / ``scann_dense_chain`` and their ``_det`` forms: the backward step list of the engine
  (LayerNorm backward with dgamma / dbeta, swish', three A operands, resid / C2 / image hand-over), training-mode
  Dropout in every mode and the no-pair fix-up, at row counts around the 32-row tile, 64-row tile and wave limits.
* Models deeper than one weight-gradient launch holds.

Bounds.  Every output of a GEMM is checked element by element: |got - ref| <= TOL * (the same sum over absolute
values: |X|^T |Y| for dW, |A| |W| + |bias| + |resid| for a chain step, carried through swish' and the Dropout mask).  A
max-relative bound would hide errors in the small entries.  LayerNorm outputs (forward and backward) keep the
max-relative TOL_OUT of test_gpu_parity.py.  TOL = 1e-5 is fp32-level; the kernels compute 3xTF32.  Worst measured
ratio of error to bound on a B200 (148 SMs, 1000 W power limit): 0.14 (weight-gradient batch), 0.12 (chain GEMM
outputs), 0.028 (dgamma / dbeta)."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from scann_b200.config import model_spec                           # noqa: E402
from scann_b200.configs import get_config                          # noqa: E402
from scann_b200.params import ParamLayout                          # noqa: E402
from scann_b200.synth import Shape, make_batch                     # noqa: E402
from tests.test_gpu_parity import CHAIN_ROWS, TOL_GRAD, TOL_OUT, chain_rows, rel   # noqa: E402

D = 128
TOL = 1e-5
f64 = np.float64


def abi():
    from scann_b200 import _abi
    _abi.require_gpu()
    return _abi


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _within(got, ref, bound, what):
    """|got - ref| <= TOL * bound element by element (exact where the bound is 0); returns the worst ratio."""
    got = np.asarray(got, f64)
    err = np.abs(got - ref)
    ok = np.isfinite(got) & (err <= TOL * bound)
    nz = bound > 0
    ratio = float((err[nz] / (TOL * bound[nz])).max()) if nz.any() else 0.0
    assert ok.all(), (what, int((~ok).sum()), ratio)
    return ratio


# ----------------------------------------------------------------------------------------------- weight-gradient batch
DENSE_CELL = Shape("dense_cell", 4, 12, 40, (5, 12), (1, 6, 7, 8, 9), None, (20, 40), (0.9, 4.0), (0.4, 3.0))
# name -> (SCANN_TILE_STRIDE, batch shape, B, tile stride of the plan)
PLANS = {"stride32": ("0", "qm9", 16, 32), "stride64": ("64", "qm9", 16, 64), "stride128": ("128", "qm9", 16, 128),
         "nbrs40": ("0", DENSE_CELL, 4, 128)}


class Plan:
    """A pair plan built by Engine.load_batch, and its valid rows on the host."""

    def __init__(self, monkeypatch, name):
        from scann_b200.engine import Engine
        pref, shape, B, stride = PLANS[name]
        monkeypatch.setenv("SCANN_TILE_STRIDE", pref)
        cfg = get_config("qm9")
        cfg["model"]["n_attention"] = 1
        spec = model_spec(cfg)
        self.eng = Engine(spec, ParamLayout(spec).randomize_arena(1))
        inputs, _ = make_batch(shape, 3, B=B)
        b = self.b = self.eng.load_batch(inputs)
        torch.cuda.synchronize()
        self.eng.check_status()
        assert b.stride == stride
        if name == "nbrs40":
            assert inputs["neighbor_mask"].sum(-1).max() > 32
        nt = int(b.ntiles.item())
        pc = b.pair_c.cpu().numpy()
        self.pair_j = b.pair_j.cpu().numpy()
        self.valid = np.zeros(b.rows, bool)
        self.valid[:nt * b.stride] = pc[:nt * b.stride] >= 0
        assert (~self.valid[:nt * b.stride]).any()           # padding rows inside the tiles: the kernel must skip them
        assert self.valid.sum() == int(b.nvalid.item())

    def args(self, compact):
        b = self.b
        if compact:
            return (b.ntiles.data_ptr(), b.stride, b.pair_c.data_ptr(), b.pair_j.data_ptr(), b.valid_rows.data_ptr(),
                    b.valid_j.data_ptr(), b.nvalid.data_ptr())
        return (b.ntiles.data_ptr(), b.stride, b.pair_c.data_ptr(), b.pair_j.data_ptr(), 0, 0, 0)


class Table:
    """A problem table with operands on the device and its fp64 restatement.  Rows the kernel must not read hold NaN."""

    def __init__(self, plan, seed):
        self.plan, self.R = plan, plan.b.R
        self.rng = np.random.default_rng(seed)
        self.keep, self.probs, self.refs = [], [], []

    def _rand(self, *shape):
        return self.rng.standard_normal(shape).astype(np.float32)

    def atom(self, rows, ldx=D, ldy=D, xoff=0, yoff=0, bias=True):
        """A per-atom problem over `rows` rows of [rows + 37, ld] buffers: columns [off, off + 128) of the first `rows`
        rows are the operand, everything else is NaN."""
        X = np.full((rows + 37, ldx), np.nan, np.float32)
        Y = np.full((rows + 37, ldy), np.nan, np.float32)
        X[:rows, xoff:xoff + D] = self._rand(rows, D)
        Y[:rows, yoff:yoff + D] = self._rand(rows, D)
        self._problem(_dev(X), 4 * xoff, ldx, _dev(Y), 4 * yoff, ldy, rows, X[:rows, xoff:xoff + D].astype(f64),
                      Y[:rows, yoff:yoff + D].astype(f64), bias)

    def pair(self, with_xg, bias=False):
        """A per-pair problem over the plan's rows (padding rows NaN); with_xg: X rows scaled by xg[pair_j[row]]."""
        p = self.plan
        X = np.full((p.b.rows, D), np.nan, np.float32)
        Y = np.full((p.b.rows, D), np.nan, np.float32)
        n = int(p.valid.sum())
        X[p.valid], Y[p.valid] = self._rand(n, D), self._rand(n, D)
        x64 = X[p.valid].astype(f64)
        xg = None
        if with_xg:
            G = self._rand(self.R, D)
            xg = _dev(G)
            x64 = x64 * G[p.pair_j[p.valid]].astype(f64)
        self._problem(_dev(X), 0, D, _dev(Y), 0, D, -1, x64, Y[p.valid].astype(f64), bias, xg)

    def _problem(self, X, xoff, ldx, Y, yoff, ldy, rows, x64, y64, bias, xg=None):
        A = abi()
        dW = torch.empty(D, D, device="cuda")
        db = torch.empty(D, device="cuda") if bias else None
        self.keep += [t for t in (X, Y, dW, db, xg) if t is not None]
        pr = A.WgradProblem()
        pr.X, pr.Y = X.data_ptr() + xoff, Y.data_ptr() + yoff
        pr.xg = xg.data_ptr() if xg is not None else None
        pr.dW, pr.db = dW.data_ptr(), db.data_ptr() if bias else None
        pr.ldx, pr.ldy, pr.rows, pr.pad = ldx, ldy, rows, 0
        self.probs.append(pr)
        self.refs.append(dict(dW=dW, db=db, ref=x64.T @ y64, abs=np.abs(x64).T @ np.abs(y64),
                              bref=y64.sum(0) if bias else None, babs=np.abs(y64).sum(0) if bias else None))

    def device(self):
        """The table as a device array: (address, problem count)."""
        arr = (abi().WgradProblem * len(self.probs))(*self.probs)
        t = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).cuda()
        self.keep.append(t)
        return t.data_ptr(), len(self.probs)

    def run(self, grid, compact, det, prefill=None):
        """One launch (det: the deterministic kernel and the reduce); returns (dW, db) of every problem on the host.
        prefill: per-problem (dW, db) host values to start from (default form), or NaN (deterministic form)."""
        A = abi()
        lib = A.lib
        for i, r in enumerate(self.refs):
            r["dW"].copy_(torch.from_numpy(prefill[i][0]) if prefill else torch.full((D, D), float("nan")))
            if r["db"] is not None:
                r["db"].copy_(torch.from_numpy(prefill[i][1]) if prefill else torch.full((D,), float("nan")))
        table, n = self.device()
        nt, stride, pc, pj, vr, vj, nv = self.plan.args(compact)
        if det:
            slots = torch.empty(grid, 2, D * D, device="cuda")
            bslots = torch.empty(grid, 2, D, device="cuda")
            A.check(lib.scann_wgrad_batch_tc_det(grid, table, n, nt, stride, pc, pj, vr, vj, nv, slots.data_ptr(),
                                                    bslots.data_ptr(), None), "wgrad_batch_tc_det")
            A.check(lib.scann_wgrad_batch_reduce(grid, table, n, nt, stride, vr, nv, slots.data_ptr(),
                                                    bslots.data_ptr(), None), "wgrad_batch_reduce")
        else:
            A.check(lib.scann_wgrad_batch_tc(grid, table, n, nt, stride, pc, pj, vr, vj, nv, None), "wgrad_batch_tc")
        torch.cuda.synchronize()
        return [(r["dW"].cpu().numpy(), None if r["db"] is None else r["db"].cpu().numpy()) for r in self.refs]

    def check(self, out, prefill=None):
        """Default form: out - prefill, with |prefill| added to the bound (one fp32 add onto it); deterministic form: out
        itself (every element stored exactly once over the NaN it started from)."""
        worst = 0.0
        for i, (r, (dW, db)) in enumerate(zip(self.refs, out)):
            p = prefill[i] if prefill else (0.0, 0.0)
            base = np.abs(np.asarray(p[0], f64))
            worst = max(worst, _within(dW - np.asarray(p[0], f64), r["ref"], r["abs"] + base, ("dW", i)))
            if r["db"] is not None:
                bb = np.abs(np.asarray(p[1], f64))
                worst = max(worst, _within(db - np.asarray(p[1], f64), r["bref"], r["babs"] + bb, ("db", i)))
        return worst


def _engine_like_table(t, B, L):
    """The engine's table for a SCANN+ model with attention normalisation (Engine._wgrad_table, 4 + 7 L problems) with
    per-atom problems of 1, 31, 32 and 33 rows and one strided left operand after the four head problems."""
    R = t.R
    t.atom(B)                                   # bf_property over the B structure rows
    t.atom(R, ldy=2 * D, yoff=0)                # GlobalAttention query: right operand = columns 0..127 of [R, 256]
    t.atom(R, ldy=2 * D, yoff=D)                # GlobalAttention key: columns 128..255
    t.atom(R)                                   # after_Lc
    for rows in (1, 31, 32, 33):
        t.atom(rows)
    t.atom(R, ldx=2 * D, xoff=D, bias=False)
    for _ in range(L):
        t.pair(True)                            # key/kernel: (x[j] * g')^T d_k
        t.pair(False)                           # filter_geo rows 128..255: g^T d_pre
        t.atom(R)                               # residual_norm dense_1
        t.atom(R)                               # residual_norm dense
        t.atom(R)                               # filter_geo rows 0..127 (+ bias)
        t.atom(R, bias=False)                   # filter_geo rows 256..383
        t.atom(R)                               # query


def _prefill(t):
    rng = np.random.default_rng(99)
    return [(rng.standard_normal((D, D)).astype(np.float32),
             rng.standard_normal(D).astype(np.float32) if r["db"] is not None else None) for r in t.refs]


@pytest.mark.parametrize("grid", ["1", "3", "sms"])
@pytest.mark.parametrize("compact", [True, False], ids=["valid_rows", "all_rows"])
@pytest.mark.parametrize("plan", list(PLANS))
def test_wgrad_batch_matches_fp64(monkeypatch, plan, compact, grid):
    """Default form: dW / db accumulated onto known values.  Deterministic form: stored over NaN, identical bits in two
    runs, and within the bound of the default form's result."""
    p = Plan(monkeypatch, plan)
    G = p.eng.la_grid if grid == "sms" else int(grid)
    t = Table(p, seed=len(plan) + 7 * G)
    _engine_like_table(t, p.b.B, 2)
    assert len(t.probs) == 4 + 5 + 7 * 2
    pre = _prefill(t)
    r_def = t.check(t.run(G, compact, False, pre), pre)
    det1 = t.run(G, compact, True)
    r_det = t.check(det1)
    det2 = t.run(G, compact, True)
    for (a, ab), (b, bb) in zip(det1, det2):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert ab is None or np.array_equal(ab.view(np.uint32), bb.view(np.uint32))
    dflt = t.run(G, compact, False, [(np.zeros((D, D), np.float32), np.zeros(D, np.float32)) for _ in t.refs])
    for r, (a, _), (b, _) in zip(t.refs, det1, dflt):
        assert (np.abs(a.astype(f64) - b) <= 2 * TOL * r["abs"]).all()
    print(f"worst error / bound: default {r_def:.3g}, deterministic {r_det:.3g}")


def test_wgrad_batch_table_limit(monkeypatch):
    """A table of scann_wgrad_batch_max_problems() problems runs in all three entry points; one more is refused."""
    lib = abi().lib
    m = lib.scann_wgrad_batch_max_problems()
    assert m >= 4 + 7 * 11                    # the deepest shipped configuration (11 layers) is one launch
    p = Plan(monkeypatch, "stride32")
    t = Table(p, seed=5)
    t.pair(True)
    t.pair(False, bias=True)
    for i in range(m - 2):
        t.atom(1 + (37 * i) % p.b.R, bias=i % 3 != 0)
    pre = _prefill(t)
    G = p.eng.la_grid
    worst = t.check(t.run(G, True, False, pre), pre)
    worst = max(worst, t.check(t.run(G, True, True)))
    print(f"worst error / bound: {worst:.3g}")
    t.atom(3)
    table, n = t.device()
    assert n == m + 1
    nt, stride, pc, pj, vr, vj, nv = p.args(True)
    slots = torch.empty(G, 2, D * D, device="cuda")
    bslots = torch.empty(G, 2, D, device="cuda")
    for call in (lambda: lib.scann_wgrad_batch_tc(G, table, n, nt, stride, pc, pj, vr, vj, nv, None),
                 lambda: lib.scann_wgrad_batch_tc_det(G, table, n, nt, stride, pc, pj, vr, vj, nv, slots.data_ptr(),
                                                      bslots.data_ptr(), None),
                 lambda: lib.scann_wgrad_batch_reduce(G, table, n, nt, stride, vr, nv, slots.data_ptr(), bslots.data_ptr(),
                                                      None)):
        assert call() != 0
        assert f"nprob must be in 1..{m}" in abi().last_error()
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------- chained Dense kernels
FORMS = ["chain2", "chain2_det", "chain", "chain_det"]


def _swish_grad(x):
    s = 1.0 / (1.0 + np.exp(-x))
    return s * (1.0 + x * (1.0 - s)), s * (1.0 + np.abs(x) * (1.0 - s))    # value, sum of the absolute terms


def _ln(v, g, b):
    mu = v.mean(1, keepdims=True)
    return (v - mu) / np.sqrt(v.var(1, keepdims=True) + 1e-6) * g + b


def _ln_backward(dy, x, g):
    """dx, dgamma, dbeta, |x_hat| of keras LayerNormalization (epsilon 1e-6)."""
    xh = (x - x.mean(1, keepdims=True)) / np.sqrt(x.var(1, keepdims=True) + 1e-6)
    inv = 1.0 / np.sqrt(x.var(1, keepdims=True) + 1e-6)
    dxh = dy * g
    dx = inv * (dxh - dxh.mean(1, keepdims=True) - xh * (dxh * xh).mean(1, keepdims=True))
    return dx, (dy * xh).sum(0), dy.sum(0), np.abs(xh)


class Chain:
    """Five weight blocks: raw [in, out] and transposed copies for scann_dense_chain, operand images (both orientations)
    for scann_dense_chain2; a Dropout control block."""

    def __init__(self, seed, form):
        A = abi()
        self.lib, self.form = A.lib, form
        self.new = form.startswith("chain2")
        self.det = form.endswith("_det")
        rng = np.random.default_rng(seed)
        self.rng = rng
        self.W = [(rng.standard_normal((D, D)) / np.sqrt(D)).astype(np.float32) for _ in range(5)]
        self.raw = _dev(np.concatenate([w.ravel() for w in self.W]))
        self.rawT = _dev(np.concatenate([w.T.ravel() for w in self.W]))
        offs = torch.arange(5, dtype=torch.int32, device="cuda") * (D * D)
        self.img = torch.zeros(5 * 2 * 32768 + 256, device="cuda")
        self.ibase = (self.img.data_ptr() + 1023) // 1024 * 1024
        A.check(self.lib.scann_weight_images(self.raw.data_ptr(), offs.data_ptr(), 5, self.ibase, None))
        self.status = torch.zeros(8, dtype=torch.int32, device="cuda")
        self.seed, self.rate = 1234567 + seed, 0.1
        from scann_b200 import dropout as dr
        scale = np.float32(1.0) / (np.float32(1.0) - np.float32(self.rate))
        self.ctl = _dev(np.array([self.seed, dr.threshold(self.rate), scale.view(np.uint32), 1], np.uint32).view(np.int32))

    def w(self, i, transposed=False):
        """W[i] (x @ W) or W[i]^T (x @ W^T) as the step's weight pointer."""
        if self.new:
            return self.ibase + (i * 2 + (1 if transposed else 0)) * 131072
        return (self.rawT if transposed else self.raw).data_ptr() + i * D * D * 4

    def mask(self, site, R):
        from scann_b200 import dropout as dr
        return dr.drop_mask(self.seed, site, R, self.rate).astype(f64)

    def grid(self, R):
        return self.lib.scann_dense_chain2_grid(R) if self.new else self.lib.scann_dense_chain_grid(R)

    def run(self, steps, R):
        A = abi()
        arr = (A.ChainStep * len(steps))(*steps)
        p = ctypes.cast(arr, ctypes.c_void_p)
        if self.new:
            fn = self.lib.scann_dense_chain2_det if self.det else self.lib.scann_dense_chain2
            A.check(fn(p, len(steps), R, self.status.data_ptr(), None), self.form)
        else:
            fn = self.lib.scann_dense_chain_det if self.det else self.lib.scann_dense_chain
            A.check(fn(p, len(steps), R, None), self.form)
        torch.cuda.synchronize()
        assert int(self.status[0].item()) == 0


def _rand(rng, *shape, scale=1.0, shift=0.0):
    return (shift + scale * rng.standard_normal(shape)).astype(np.float32)


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("rows", CHAIN_ROWS)
def test_chain_backward_steps_match_fp64(form, rows):
    """The tail of a backward layer as Engine._backward_chained builds it: [s_pre | t_sc | dq] @ [W0 | W1 | W2]^T + dx_sc
    -> LayerNorm backward of the ResidualNorm (dgamma / dbeta; C = d_v2, C2 and the image = d_v2 * Dropout mask) ->
    @ W3^T * swish'(t1) -> @ W4^T + d_v2 -> LayerNorm backward of the attention output (C and C2)."""
    from scann_b200._abi import chain_step
    R = chain_rows(rows)
    c = Chain(R % 1000 + 3, form)
    rng = c.rng
    sp, ts, dq, dxs, v2, t1, cp = (_rand(rng, R, D) for _ in range(7))
    g1, g2 = _rand(rng, D, scale=0.1, shift=1.0), _rand(rng, D, scale=0.1, shift=1.0)
    d = {k: _dev(v) for k, v in dict(sp=sp, ts=ts, dq=dq, dxs=dxs, v2=v2, t1=t1, cp=cp, g1=g1, g2=g2).items()}
    out = {k: torch.full((R, D), float("nan"), device="cuda") for k in ("d_v2", "d_v2m", "d_t1", "d_ctx", "dq_out")}
    G = c.grid(R)
    pre = _rand(rng, 4, D)                              # default form: dgamma / dbeta accumulate onto these
    ln = torch.full((4, G, D), float("nan"), device="cuda") if c.det else _dev(pre)
    lnp = [ln[i].data_ptr() for i in range(4)]
    site = 3
    steps = [
        chain_step(A=[d["sp"].data_ptr(), d["ts"].data_ptr(), d["dq"].data_ptr()], W=[c.w(0, True), c.w(1, True), c.w(2, True)],
                   resid=d["dxs"].data_ptr(), mode=4, pre_in=d["v2"].data_ptr(), gamma=d["g1"].data_ptr(), dgamma=lnp[0],
                   dbeta=lnp[1], C_=out["d_v2"].data_ptr(), C2=out["d_v2m"].data_ptr(), to_image=True,
                   drop=c.ctl.data_ptr(), drop_site=site),
        chain_step(W=[c.w(3, True)], mode=2, pre_in=d["t1"].data_ptr(), C_=out["d_t1"].data_ptr(), to_image=True),
        chain_step(W=[c.w(4, True)], resid=out["d_v2"].data_ptr(), mode=4, pre_in=d["cp"].data_ptr(), gamma=d["g2"].data_ptr(),
                   dgamma=lnp[2], dbeta=lnp[3], C_=out["d_ctx"].data_ptr(), C2=out["dq_out"].data_ptr()),
    ]

    def once():
        if c.det:
            ln.fill_(float("nan"))
        else:
            ln.copy_(torch.from_numpy(pre))
        for t in out.values():
            t.fill_(float("nan"))
        c.run(steps, R)
        return {k: v.cpu().numpy() for k, v in out.items()}, ln.cpu().numpy()

    got, lng = once()
    W = [w.astype(f64) for w in c.W]
    aW = [np.abs(w) for w in W]
    A = [x.astype(f64) for x in (sp, ts, dq)]
    V0 = A[0] @ W[0].T + A[1] @ W[1].T + A[2] @ W[2].T + dxs
    a0 = np.abs(A[0]) @ aW[0].T + np.abs(A[1]) @ aW[1].T + np.abs(A[2]) @ aW[2].T + np.abs(dxs)
    dx0, dg1, db1, xh1 = _ln_backward(V0, v2.astype(f64), g1.astype(f64))
    m = c.mask(site, R)
    V1 = (dx0 * m) @ W[3].T
    sg, sa = _swish_grad(t1.astype(f64))
    o1, a1 = V1 * sg, (np.abs(dx0 * m) @ aW[3].T) * sa
    V2 = o1 @ W[4].T + dx0
    a2 = a1 @ aW[4].T + np.abs(dx0)
    dx2, dg2, db2, xh2 = _ln_backward(V2, cp.astype(f64), g2.astype(f64))
    assert rel(got["d_v2"], dx0) <= TOL_OUT
    assert rel(got["d_v2m"], dx0 * m) <= TOL_OUT and (got["d_v2m"][m == 0] == 0).all()
    assert rel(got["d_ctx"], dx2) <= TOL_OUT
    assert np.array_equal(got["dq_out"], got["d_ctx"])
    worst = _within(got["d_t1"], o1, a1, "d_t1")
    # deterministic form: the slots of the CTAs, summed here; default form: accumulated onto `pre` (one more fp32 add)
    sums, base = (lng.astype(f64).sum(1), np.zeros((4, D))) if c.det else (lng.astype(f64) - pre, np.abs(pre.astype(f64)))
    wln = 0.0
    for i, (ref, bound) in enumerate(((dg1, (a0 * xh1).sum(0)), (db1, a0.sum(0)), (dg2, (a2 * xh2).sum(0)),
                                      (db2, a2.sum(0)))):
        wln = max(wln, _within(sums[i], ref, bound + base[i], ("dgamma / dbeta", i)))
    if c.det:
        got2, lng2 = once()
        assert np.array_equal(lng.view(np.uint32), lng2.view(np.uint32))
        for k in got:
            assert np.array_equal(got[k].view(np.uint32), got2[k].view(np.uint32)), k
    print(f"worst error / bound: d_t1 {worst:.3g}, dgamma / dbeta {wln:.3g}")


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("rows", CHAIN_ROWS)
def test_chain_forward_dropout_and_no_pair_rows_match_fp64(form, rows):
    """ResidualNorm with Dropout after both Dense layers (modes 1 and 3), then the next layer's projections from the
    resident image into one [R, 384] buffer: mode 0 with Dropout, mode 2 with Dropout, and the query with the no-pair
    fix-up (rows with cnt == 0 also get np_ctx = q and np_out = LayerNorm(q); the others are not written)."""
    from scann_b200._abi import chain_step
    R = chain_rows(rows)
    c = Chain(R % 1000 + 11, form)
    rng = c.rng
    x, pp = _rand(rng, R, D), _rand(rng, R, D)
    b = [_rand(rng, D, scale=0.1) for _ in range(5)]
    g, be = _rand(rng, D, scale=0.1, shift=1.0), _rand(rng, D, scale=0.1)
    g2, be2 = _rand(rng, D, scale=0.1, shift=1.0), _rand(rng, D, scale=0.1)
    cnt = rng.integers(0, 4, R).astype(np.int32)
    cnt[::5] = 0
    d = {k: _dev(v) for k, v in dict(x=x, pp=pp, g=g, be=be, g2=g2, be2=be2, cnt=cnt).items()}
    bd = [_dev(v) for v in b]
    out = {k: torch.full((R, D), float("nan"), device="cuda") for k in ("t1", "h1", "v2", "x1", "np_ctx", "np_out")}
    proj = torch.full((R, 3 * D), float("nan"), device="cuda")
    P = lambda t, off=0: t.data_ptr() + 4 * off                                              # noqa: E731
    sites = (5, 6, 7, 8)
    steps = [
        chain_step(A=[P(d["x"])], W=[c.w(0)], bias=P(bd[0]), mode=1, pre_out=P(out["t1"]), C_=P(out["h1"]), to_image=True,
                   drop=P(c.ctl), drop_site=sites[0]),
        chain_step(W=[c.w(1)], bias=P(bd[1]), resid=P(d["x"]), mode=3, pre_out=P(out["v2"]), gamma=P(d["g"]),
                   beta=P(d["be"]), C_=P(out["x1"]), to_image=True, drop=P(c.ctl), drop_site=sites[1]),
        chain_step(W=[c.w(2)], bias=P(bd[2]), C_=P(proj), ldc=3 * D, drop=P(c.ctl), drop_site=sites[2]),
        chain_step(W=[c.w(3)], mode=2, pre_in=P(d["pp"]), C_=P(proj, D), ldc=3 * D, drop=P(c.ctl), drop_site=sites[3]),
        chain_step(W=[c.w(4)], bias=P(bd[4]), C_=P(proj, 2 * D), ldc=3 * D, cnt=P(d["cnt"]), np_ctx=P(out["np_ctx"]),
                   np_out=P(out["np_out"]), gamma=P(d["g2"]), beta=P(d["be2"])),
    ]
    c.run(steps, R)
    got = {k: v.cpu().numpy() for k, v in out.items()}
    pj = proj.cpu().numpy()
    W = [w.astype(f64) for w in c.W]
    aW = [np.abs(w) for w in W]
    B = [v.astype(f64) for v in b]
    X = x.astype(f64)
    m = [c.mask(s, R) for s in sites]
    V0 = (X @ W[0] + B[0]) * m[0]
    a0 = (np.abs(X) @ aW[0] + np.abs(B[0])) * m[0]
    h1 = V0 / (1.0 + np.exp(-V0))
    V1 = (h1 @ W[1] + B[1]) * m[1] + X
    a1 = (np.abs(h1) @ aW[1] + np.abs(B[1])) * m[1] + np.abs(X)
    x1 = _ln(V1, g.astype(f64), be.astype(f64))
    ax1 = np.abs(x1)
    P0, a2 = (x1 @ W[2] + B[2]) * m[2], (ax1 @ aW[2] + np.abs(B[2])) * m[2]
    sg, sa = _swish_grad(pp.astype(f64))
    P1, a3 = (x1 @ W[3]) * m[3] * sg, (ax1 @ aW[3]) * m[3] * sa
    P2, a4 = x1 @ W[4] + B[4], ax1 @ aW[4] + np.abs(B[4])
    worst = max(_within(got["t1"], V0, a0, "t1 (mode 1 pre_out)"), _within(got["v2"], V1, a1, "v2 (mode 3 pre_out)"),
                _within(pj[:, :D], P0, a2, "mode 0"), _within(pj[:, D:2 * D], P1, a3, "mode 2"),
                _within(pj[:, 2 * D:], P2, a4, "query"))
    assert rel(got["h1"], h1) <= TOL_OUT
    assert rel(got["x1"], x1) <= TOL_OUT
    nop = cnt == 0
    worst = max(worst, _within(got["np_ctx"][nop], P2[nop], a4[nop], "np_ctx"))
    assert rel(got["np_out"][nop], _ln(P2[nop], g2.astype(f64), be2.astype(f64))) <= TOL_OUT
    assert np.isnan(got["np_ctx"][~nop]).all() and np.isnan(got["np_out"][~nop]).all()
    print(f"worst error / bound: {worst:.3g}")


# ----------------------------------------------------------------------------------------------- deep models
@pytest.mark.parametrize("L", [14, 20])
def test_deep_models_train_and_predict(monkeypatch, L):
    """SCANN+ deeper than one weight-gradient launch holds (4 + 7 L problems): the table is cut into launches of at most
    scann_wgrad_batch_max_problems() problems; the per-layer weight-gradient kernels (SCANN_WGRAD_BATCH=0) train the
    same model; predict with every layer's local-attention scores works at this depth."""
    from oracle import scann_oracle as O
    from scann_b200.engine import Engine
    from scann_b200.model import create_model
    from tests.golden.make_golden import oracle_kwargs
    from tests.test_local_attention import check_against_oracle
    lib = abi().lib
    cfg = get_config("qm9")
    cfg["model"]["n_attention"] = L
    spec = model_spec(cfg)
    lay = ParamLayout(spec)
    arena = lay.randomize_arena(21)
    inputs, target = make_batch("qm9", 13, B=4)
    w = lay.to_dict(arena)
    eng = Engine(spec, arena)
    b = eng.load_batch(inputs)
    eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3, apply=False, want_grads=True)
    torch.cuda.synchronize()
    eng.check_status()
    launches = eng._wgrad_table(b, eng._workspace(b, True))
    m = lib.scann_wgrad_batch_max_problems()
    assert [n for _, n in launches] == [min(m, 4 + 7 * L - i) for i in range(0, 4 + 7 * L, m)]
    assert len(launches) > 1
    batched = eng.grad_out.cpu().numpy().astype(f64)
    monkeypatch.setenv("SCANN_WGRAD_BATCH", "0")
    eng0 = Engine(spec, arena)
    assert not eng0.use_wgrad_batch
    b0 = eng0.load_batch(inputs)
    eng0.train_step(b0, torch.from_numpy(target).cuda(), lr=1e-3, apply=False, want_grads=True)
    torch.cuda.synchronize()
    eng0.check_status()
    l2n = [e.name for e in lay if e.l2]
    # the bounds of test_full_configuration_parity_against_oracle: 1e-5 / 1e-4, or 5 x the distance of the reference's
    # own fp32 arithmetic from fp64 where that is larger
    loss, y_ref, ga_ref, grads = O.loss_and_grads(w, inputs, target, l2n, **oracle_kwargs(spec))
    _, y32, ga32, grads32 = O.loss_and_grads(w, inputs, target, l2n, dtype=torch.float32, **oracle_kwargs(spec))
    gmax = max(np.abs(v).max() for v in grads.values())
    g0 = lay.to_dict(eng0.grad_out.cpu().numpy())
    g1 = lay.to_dict(batched)
    for e in lay:
        ref = grads[e.name]
        noise32 = np.abs(grads32[e.name].astype(f64) - ref).max()
        bound = max(TOL_GRAD * max(np.abs(ref).max(), 1e-2 * gmax), 5.0 * noise32)
        assert np.abs(g0[e.name] - ref).max() <= bound, (e.name, "SCANN_WGRAD_BATCH=0")
        assert np.abs(g1[e.name] - ref).max() <= bound, (e.name, "batched")
    model = create_model(cfg, infer=True, arena=arena)
    y, ga, la = model.predict(inputs, local_attention=True)
    assert rel(np.asarray(y).ravel(), y_ref.ravel()) <= max(TOL_OUT, 5.0 * rel(y32, y_ref))
    assert rel(np.asarray(ga)[..., 0], ga_ref[..., 0]) <= max(TOL_OUT, 5.0 * rel(ga32, ga_ref))
    check_against_oracle(la, inputs, spec, w, full_depth=True)

