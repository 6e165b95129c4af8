"""Deterministic training mode on the GPU: bitwise-reproducible train steps, unchanged accuracy, loud refusals."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import scann_oracle as O                               # noqa: E402
from scann_b200.config import model_spec                           # noqa: E402
from scann_b200.configs import get_config                          # noqa: E402
from scann_b200.params import ParamLayout                          # noqa: E402
from scann_b200.synth import make_batch                            # noqa: E402
from tests.golden.make_golden import CASES, build_case, oracle_kwargs   # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_GRAD = 1e-4

NOUP = {"g_update": False, "gaussian_d": 4.0}      # model_ptgp.yaml lacks these two keys (as in bench.py)
# name -> (config, batch shape, B, layers, model overrides, training-mode Dropout, feature)
REPRO = {
    "qm9_b128_l7_dropout": ("qm9", "qm9", 128, 7, {}, True, "atomic"),
    "mp2018_b64_l4": ("mp2018", "mp2018", 64, 4, {}, False, "atomic"),
    "fullerene_b128_l7": ("fullerene", "fullerene", 128, 7, {}, False, "atomic"),
    "qm9_ring_b16_l2": ("qm9", "qm9", 16, 2, {"use_ring": True}, False, "atomic"),
    # g_update=False, ring features: the g_update=False attention / filter backward
    "ptgp_b16_l3": ("ptgp", "ptgp", 16, 3, NOUP, False, "atomic"),
    # 16 384 atom rows: more than one wave of the warp-specialised chained kernel, so the round-1 chained kernel runs
    "ptgp_b64_l2_round1_chain": ("ptgp", "ptgp", 64, 2, NOUP, False, "atomic"),
    "cgcnn_ring_b16_l2": ("qm9", "qm9", 16, 2, {"use_ring": True}, False, "cgcnn"),
    # deeper than one weight-gradient launch holds (4 + 7 L problems): two launches, each with its own reduce
    "qm9_b4_l14": ("qm9", "qm9", 4, 14, {}, False, "atomic"),
    "qm9_b4_l20": ("qm9", "qm9", 4, 20, {}, False, "atomic"),
}


def _spec(cfg_name, L, over, feature="atomic"):
    cfg = get_config(cfg_name, feature=feature)
    cfg["model"]["n_attention"] = L
    cfg["model"].update(over)
    spec = model_spec(cfg)
    return spec, ParamLayout(spec)


def _engine(spec, arena, **kw):
    from scann_b200.engine import Engine
    return Engine(spec, arena, deterministic=True, **kw)


def _bits(t):
    return np.ascontiguousarray(t.detach().cpu().numpy()).view(np.uint32).copy()


def _run(spec, arena, batches, dropout=False, graphs=True):
    """Train steps on a fresh deterministic engine; returns the uint32 views of everything the step produces."""
    eng = _engine(spec, arena)
    eng.train_dropout = dropout
    eng.use_graphs = graphs
    losses = []
    for inputs, target in batches:
        b = eng.load_batch(inputs)
        eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3, want_grads=True)
        losses.append(_bits(eng.loss_value(b.B)))
    torch.cuda.synchronize()
    eng.check_status()
    out = {"params": _bits(eng.params), "m": _bits(eng.adam_m), "v": _bits(eng.adam_v), "grads": _bits(eng.grads),
           "grad_out": _bits(eng.grad_out), "loss": np.stack(losses)}
    del eng
    return out


def _assert_same(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _batches(shape, B, n, seed, ring=False, feature="atomic"):
    return [make_batch(shape, seed + i, B=B, use_ring=ring, feature=feature) for i in range(n)]


@pytest.mark.parametrize("name", list(REPRO))
def test_two_engines_give_identical_bits(name):
    cfg_name, shape, B, L, over, drop, feature = REPRO[name]
    spec, lay = _spec(cfg_name, L, over, feature)
    arena = lay.randomize_arena(7)
    batches = _batches(shape, B, 3, 40, ring=spec.use_ring, feature=feature)
    a = _run(spec, arena, batches, dropout=drop)
    b = _run(spec, arena, batches, dropout=drop)
    _assert_same(a, b)
    assert np.isfinite(a["params"].view(np.float32)).all()


def _hub_batch(seed):
    """Hundreds of pairs point at one atom row; duplicate neighbours and self-neighbours elsewhere."""
    inputs, target = make_batch("qm9", seed, B=16)
    nb, nm = inputs["neighbors"].copy(), inputs["neighbor_mask"].copy()
    h = int(np.argmax(inputs["atom_mask"][:, :, 0].sum(1)))        # the largest structure is the hub
    d, s = (h + 1) % 16, (h + 2) % 16
    nm[h, :, :] = inputs["atom_mask"][h, :, 0][:, None]          # every real atom uses all 16 slots
    nb[h, :, :] = 0                                               # ... and every one of them points at atom 0
    nb[d, :, ::2] = nb[d, :, 1::2]                                # duplicates
    nb[s, :, 0] = np.arange(nb.shape[1])                          # self
    inputs = dict(inputs, neighbors=np.where(nm, nb, 0).astype(np.int32), neighbor_mask=nm)
    return inputs, target


def test_hub_batch_five_steps():
    spec, lay = _spec("qm9", 3, {})
    arena = lay.randomize_arena(8)
    inputs, target = _hub_batch(5)
    h = int(np.argmax(inputs["atom_mask"][:, :, 0].sum(1)))
    assert int((inputs["neighbor_mask"][h] & (inputs["neighbors"][h] == 0)).sum()) >= 200   # pairs into one atom row
    batches = [(inputs, target)] * 5
    _assert_same(_run(spec, arena, batches), _run(spec, arena, batches))


def test_graph_replay_and_eager_steps_agree():
    spec, lay = _spec("qm9", 3, {})
    arena = lay.randomize_arena(9)
    batches = _batches("qm9", 64, 3, 50)
    _assert_same(_run(spec, arena, batches, graphs=True), _run(spec, arena, batches, graphs=False))


_CHILD = r"""
import hashlib, sys
import numpy as np, torch
sys.path.insert(0, {root!r})
from scann_b200.config import model_spec
from scann_b200.configs import get_config
from scann_b200.engine import Engine
from scann_b200.params import ParamLayout
from scann_b200.synth import make_batch
cfg = get_config("qm9"); cfg["model"]["n_attention"] = 3
spec = model_spec(cfg); lay = ParamLayout(spec)
eng = Engine(spec, lay.randomize_arena(10), deterministic=True)
for i in range(3):
    inputs, target = make_batch("qm9", 60 + i, B=64)
    b = eng.load_batch(inputs)
    eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3)
torch.cuda.synchronize()
print(hashlib.sha256(eng.params.cpu().numpy().tobytes()).hexdigest())
"""


def test_fresh_process_gives_the_same_parameters():
    spec, lay = _spec("qm9", 3, {})
    here = _run(spec, lay.randomize_arena(10), _batches("qm9", 64, 3, 60))
    env = dict(os.environ, PYTHONNOUSERSITE="1")
    env.pop("SCANN_DETERMINISTIC", None)
    out = subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT)], capture_output=True, text=True, env=env,
                         timeout=600)
    assert out.returncode == 0, out.stderr
    assert out.stdout.strip().splitlines()[-1] == hashlib.sha256(here["params"].tobytes()).hexdigest()


@pytest.mark.parametrize("shape,B,hub", [("qm9", 128, False), ("mp2018", 64, False), ("qm9", 16, True)])
def test_inverse_csr_is_a_stable_argsort(shape, B, hub):
    spec, lay = _spec("qm9", 2, {})
    eng = _engine(spec, lay.randomize_arena(1))
    inputs = _hub_batch(3)[0] if hub else make_batch(shape, 2, B=B)[0]
    b = eng.load_batch(inputs)
    torch.cuda.synchronize()
    pc, pj = b.pair_c.cpu().numpy(), b.pair_j.cpu().numpy()
    rows = np.flatnonzero(pc >= 0)
    order = np.argsort(pj[rows], kind="stable")
    want_idx = rows[order]
    want_ptr = np.concatenate([[0], np.cumsum(np.bincount(pj[rows], minlength=b.R))])
    ptr = b.inv_ptr.cpu().numpy()
    assert np.array_equal(ptr, want_ptr)
    assert np.array_equal(b.inv_idx.cpu().numpy()[:ptr[-1]], want_idx)


def _oracle_kwargs(spec):
    return dict(oracle_kwargs(spec), use_ring=True) if spec.use_ring else oracle_kwargs(spec)


def _det_train(spec, arena, inputs, target):
    eng = _engine(spec, arena)
    b = eng.load_batch(inputs)
    eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3, apply=False, want_grads=True)
    torch.cuda.synchronize()
    eng.check_status()
    ws = eng._workspace(b, True)
    return (eng.loss_value(b.B).cpu().numpy(), eng.grad_out.cpu().numpy().astype(np.float64), ws["y"].cpu().numpy(),
            ws["ga"].cpu().numpy().reshape(b.B, b.M))


@pytest.mark.parametrize("name", list(CASES))
def test_golden_cases_keep_their_accuracy(name):
    """The bounds test_gpu_parity.py applies to the default engine on the committed golden cases."""
    from tests.test_gpu_parity import TOL_GRAD as PTOL, GOLDEN, ga_tolerance, golden_y_tolerance, rel
    cfg, spec, lay, arena, inputs, target = build_case(name)
    z = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    lv, g, y, ga = _det_train(spec, arena, inputs, target)
    assert rel(y, z["y"].ravel()) <= golden_y_tolerance(name)
    assert rel(ga, z["ga"][..., 0]) <= ga_tolerance(spec, lay, arena, inputs)
    assert abs(lv[0] - float(z["loss"])) <= 1e-5 * abs(float(z["loss"]))
    assert rel(g[z["grad_idx"]], z["grad_sample"]) <= PTOL
    assert abs(np.sqrt((g ** 2).sum()) - float(z["grad_l2norm"])) <= PTOL * float(z["grad_l2norm"])


# the full-configuration cases of test_gpu_parity.py that the deterministic mode trains
FULL = {"qm9_b128_l7": ("qm9", "qm9", 128, {}), "ptgp_b16_l11": ("ptgp", "ptgp", 16, NOUP),
        "qm9_b352_l2": ("qm9", "qm9", 352, {"n_attention": 2}), "ptgp_b64_l2": ("ptgp", "ptgp", 64, dict(NOUP, n_attention=2))}


@pytest.mark.parametrize("name", list(FULL))
def test_full_configuration_keeps_its_accuracy(name):
    """Full depth: outputs, ga_score, loss and every per-tensor gradient against the fp64 oracle, with the bounds
    test_full_configuration_parity_against_oracle applies to the default engine."""
    from scann_b200._abi import lib
    from tests.test_gpu_parity import ROUND1_CHAIN, TOL_GRAD as PTOL, TOL_OUT, rel
    cfg_name, shape, B, over = FULL[name]
    cfg = get_config(cfg_name)
    cfg["model"].update(over)
    spec = model_spec(cfg)
    lay = ParamLayout(spec)
    arena = lay.randomize_arena(21)
    ring = bool(spec.use_ring)
    inputs, target = make_batch(shape, 13, B=B, use_ring=ring)
    if name in ROUND1_CHAIN:
        assert B * inputs["atomic"].shape[1] > lib.scann_dense_chain2_max_rows()
    w = lay.to_dict(arena)
    l2n = [e.name for e in lay if e.l2]
    kw = _oracle_kwargs(spec)
    loss, y_ref, ga_ref, grads = O.loss_and_grads(w, inputs, target, l2n, **kw)
    loss32, y32, ga32, grads32 = O.loss_and_grads(w, inputs, target, l2n, dtype=torch.float32, **kw)
    FULL_NOISE = 5.0
    lv, g, y, ga = _det_train(spec, arena, inputs, target)
    assert rel(y, y_ref.ravel()) <= max(TOL_OUT, FULL_NOISE * rel(y32, y_ref))
    assert rel(ga, ga_ref[..., 0]) <= max(TOL_OUT, FULL_NOISE * rel(ga32, ga_ref))
    assert abs(lv[0] - float(loss)) <= 1e-5 * abs(float(loss))
    g = lay.to_dict(g)
    gmax = max(np.abs(v).max() for v in grads.values())
    for e in lay:
        ref = grads[e.name]
        err = np.abs(g[e.name] - ref).max()
        noise32 = np.abs(grads32[e.name].astype(np.float64) - ref).max()
        assert err <= max(PTOL * max(np.abs(ref).max(), 1e-2 * gmax), FULL_NOISE * noise32), (e.name, err, noise32)


def test_facade_fit_twice_with_tf_deterministic_ops(monkeypatch):
    from scann_b200.datagenerator import DataIterator, synthetic_ragged
    from scann_b200.model import create_model
    monkeypatch.setenv("TF_DETERMINISTIC_OPS", "1")
    cfg = get_config("qm9")
    cfg["model"]["n_attention"] = 3
    de, dn = synthetic_ragged(96, seed=3)

    def once():
        np.random.seed(123)
        m = create_model(cfg, seed=4)
        assert m.engine.deterministic
        it = DataIterator(de, dn, batch_size=32, shuffle=True, g_update=True)
        hist = m.fit(it, epochs=2, verbose=0)
        return [np.asarray(x) for x in m.get_weights()], hist.history

    w1, h1 = once()
    w2, h2 = once()
    assert len(w1) == len(w2) and all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(w1, w2))
    assert h1 == h2


@pytest.mark.parametrize("env", [{"SCANN_ENGINE": "simt"}, {"SCANN_CHAIN": "0"}, {"SCANN_CHAIN2": "0"},
                                 {"SCANN_WGRAD_BATCH": "0"}, {"SCANN_LA_PIPE": "3"}, {"SCANN_NOUP_PIPE": "0"}])
def test_unsupported_engine_settings_are_refused(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    spec, lay = _spec("qm9", 2, {})
    eng = _engine(spec, lay.randomize_arena(1))
    inputs, target = make_batch("qm9", 1, B=8)
    b = eng.load_batch(inputs)
    with pytest.raises(NotImplementedError):
        eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3)


def test_more_than_32_neighbours_is_refused():
    spec, lay = _spec("qm9", 2, {})
    eng = _engine(spec, lay.randomize_arena(1))
    inputs, target = make_batch("qm9", 1, B=4)
    pad = lambda a: np.concatenate([a, np.zeros(a.shape[:2] + (24,), a.dtype)], axis=2)   # noqa: E731
    inputs = dict(inputs, **{k: pad(inputs[k]) for k in ("neighbors", "neighbor_mask", "neighbor_weight",
                                                          "neighbor_distance")})
    inputs["neighbor_mask"][0, 0, :] = True
    b = eng.load_batch(inputs)
    with pytest.raises(NotImplementedError, match="32"):
        eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3)


def test_default_mode_is_untouched(monkeypatch):
    monkeypatch.delenv("SCANN_DETERMINISTIC", raising=False)
    monkeypatch.delenv("TF_DETERMINISTIC_OPS", raising=False)
    from scann_b200.engine import Engine
    spec, lay = _spec("qm9", 2, {})
    eng = Engine(spec, lay.randomize_arena(1))
    assert eng.deterministic is False
    inputs, target = make_batch("qm9", 1, B=8)
    b = eng.load_batch(inputs)
    eng.train_step(b, torch.from_numpy(target).cuda(), lr=1e-3)
    torch.cuda.synchronize()
    assert b.inv_ptr is None and "pairbuf" not in eng._workspace(b, True)


_DP_CHILD = r"""
import hashlib, os, sys
import numpy as np, torch
sys.path.insert(0, {root!r})
from scann_b200 import dist as sdist
from scann_b200.configs import get_config
from scann_b200.model import create_model
from scann_b200.synth import make_batch
rank, local_rank, world = sdist.init()
torch.cuda.set_device(local_rank)
cfg = get_config("qm9"); cfg["model"]["n_attention"] = 2
m = create_model(cfg, seed=3, deterministic=True)
sdist.attach(m, world)
assert m.engine.p2p is not None
for step in range(3):
    inp, tgt = make_batch("qm9", 200 + step, B=8 * world)
    lo, hi = rank * 8, (rank + 1) * 8
    m.train_on_batch({{k: v[lo:hi] for k, v in inp.items()}}, tgt[lo:hi])
torch.cuda.synchronize()
h = hashlib.sha256(m.engine.params.cpu().numpy().tobytes() + m.engine.loss_out.cpu().numpy().tobytes()).hexdigest()
print("RANK", rank, h, flush=True)
"""


def test_two_gpu_peer_memory_runs_give_identical_bits(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    import socket
    script = tmp_path / "det_dp.py"
    script.write_text(_DP_CHILD.format(root=ROOT))
    env = dict(os.environ, SCANN_P2P_REDUCE="1")
    outs = []
    for _ in range(2):
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", str(port), str(script)]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
        outs.append(sorted(line.split()[1:] for line in res.stdout.splitlines() if line.startswith("RANK")))
    assert len(outs[0]) == 2 and outs[0] == outs[1]
    assert outs[0][0][1] == outs[0][1][1]              # the ranks agree with each other as well
