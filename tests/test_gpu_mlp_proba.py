"""GPU class probabilities of the 2-layer MLP (uml_mlp_predict_proba / predictors.mlp_predict_proba).

Yardstick: torch's own fp32 forward.  Its distance to the float64 softmax depends on the rows (4e-7 on the golden
digits rows, 7e-6 on 0..255 pixel rows, 5e-8 on standard-normal rows on the golden weights), so every batch is held to
``max |p_device - p_f64| <= max(4 * max |p_torch - p_f64|, 1e-6)`` and every row must sum to 1 within 1e-6.
"""
import numpy as np
import pandas as pd
import pytest
import torch

from oracle import mlp as omlp

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from tests.conftest import GOLDEN  # noqa: E402

ROWS = [1, 127, 128, 129, 5000, 250_001]


@pytest.fixture(scope="module")
def engine():
    from unionml_b200.engine import Engine

    return Engine(0)


@pytest.fixture(scope="module")
def golden():
    z = np.load(GOLDEN / "mlp_64_32_10.npz")
    return {k: z[k] for k in z.files}


def _weights(g):
    return g["w1"], g["b1"], g["w2"], g["b2"]


def proba_f64(X, w1, b1, w2, b2):
    """float64 softmax of the float64 logits of the float32-cast features."""
    z = omlp.logits(X, w1, b1, w2, b2, np.float64)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return e / e.sum(axis=1, keepdims=True)


def proba_torch(X, w1, b1, w2, b2):
    """PytorchModel.forward on the CPU in float32."""
    t = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)) for a in (X, w1, b1, w2, b2)]
    with torch.no_grad():
        h = torch.relu(torch.nn.functional.linear(t[0], t[1], t[2]))
        return torch.softmax(torch.nn.functional.linear(h, t[3], t[4]), dim=1).numpy()


def assert_within_criterion(p, X, w):
    ref = proba_f64(X, *w)
    tol = max(4.0 * float(np.abs(proba_torch(X, *w) - ref).max()), 1e-6)
    err = float(np.abs(p.astype(np.float64) - ref).max())
    assert err <= tol, f"max |p - p_f64| = {err:.3g} > {tol:.3g}"
    assert float(np.abs(p.astype(np.float64).sum(axis=1) - 1.0).max()) <= 1e-6


def _int_rows(rows, F=64, seed=None, hi=17):
    return np.random.default_rng(rows if seed is None else seed).integers(0, hi, size=(rows, F)).astype(np.float32)


def _normal_rows(rows, F=64, seed=None):
    return np.random.default_rng(10_000 + rows if seed is None else seed).standard_normal((rows, F)).astype(np.float32)


def test_golden_fixture(engine, golden):
    w = _weights(golden)
    m = engine.load_mlp(*w)
    p, st = engine.predict_mlp_proba(m, engine.stage(golden["X"]))
    assert p.dtype == np.float32 and p.shape == (golden["X"].shape[0], 10)
    assert st["path"] == 5 and st["n_flagged"] == 0 and st["kernel_launches"] == 2
    assert_within_criterion(p, golden["X"], w)


@pytest.mark.parametrize("rows", ROWS)
def test_tile_edges_on_every_path(engine, golden, rows, monkeypatch):
    w = _weights(golden)
    m = engine.load_mlp(*w)
    Xi, Xf = _int_rows(rows), _normal_rows(rows)
    p, st = engine.predict_mlp_proba(m, engine.stage(Xi))
    assert st["path"] == 5 and st["n_flagged"] == 0
    assert_within_criterion(p, Xi, w)
    p, st = engine.predict_mlp_proba(m, engine.stage(Xf))
    assert st["path"] == 3 and st["n_flagged"] == 0
    assert_within_criterion(p, Xf, w)
    monkeypatch.setenv("UML_B200_MLP_TC", "0")
    p, st = engine.predict_mlp_proba(m, engine.stage(Xi))
    assert st["path"] == 3
    assert_within_criterion(p, Xi, w)
    # forced onto the tensor cores, rows that are not tf32 values are all flagged and recomputed in fp64
    monkeypatch.setenv("UML_B200_MLP_TC", "1")
    p, st = engine.predict_mlp_proba(m, engine.stage(Xf))
    assert st["path"] == 5 and st["n_flagged"] == rows
    assert_within_criterion(p, Xf, w)


def test_mixed_batch_flags_exactly_the_planted_rows(engine, golden, monkeypatch):
    w = _weights(golden)
    m = engine.load_mlp(*w)
    rng = np.random.default_rng(12)
    X = _int_rows(200_000, seed=13)
    dirty = rng.choice(200_000, size=3_001, replace=False)
    X[dirty, rng.integers(0, 64, size=dirty.size)] += np.float32(1.0 / 3.0)  # not representable in 10 mantissa bits
    monkeypatch.setenv("UML_B200_MLP_TC", "1")
    p, st = engine.predict_mlp_proba(m, engine.stage(X))
    assert st["path"] == 5 and st["n_flagged"] == dirty.size
    assert_within_criterion(p, X, w)


@pytest.mark.parametrize("H", [16, 32])
@pytest.mark.parametrize("C", [2, 3, 10])
def test_tensor_core_shapes(engine, H, C):
    F = 50
    rng = np.random.default_rng(F * 1000 + H * 10 + C)
    w = ((rng.standard_normal((H, F)) * 0.2).astype(np.float32), rng.standard_normal(H).astype(np.float32),
         rng.standard_normal((C, H)).astype(np.float32), rng.standard_normal(C).astype(np.float32))
    X = rng.integers(-8, 9, size=(70_001, F)).astype(np.float32)
    p, st = engine.predict_mlp_proba(engine.load_mlp(*w), engine.stage(X))
    assert st["path"] == 5 and p.shape == (70_001, C)
    assert_within_criterion(p, X, w)


@pytest.mark.parametrize("shape", [(200, 48, 10), (64, 48, 10), (13, 20, 40)])
def test_generic_shapes_take_the_fp64_kernel(engine, shape):
    F, H, C = shape
    rng = np.random.default_rng(F + H + C)
    w = ((rng.standard_normal((H, F)) * 0.2).astype(np.float32), rng.standard_normal(H).astype(np.float32),
         rng.standard_normal((C, H)).astype(np.float32), rng.standard_normal(C).astype(np.float32))
    X = rng.integers(0, 17, size=(30_001, F)).astype(np.float32)
    p, st = engine.predict_mlp_proba(engine.load_mlp(*w), engine.stage(X))
    assert st["path"] == 2 and st["n_flagged"] == 0
    assert_within_criterion(p, X, w)


@pytest.mark.parametrize("kind", ["int", "normal"])
def test_argmax_of_probabilities_matches_the_labels(engine, golden, kind):
    w = _weights(golden)
    m = engine.load_mlp(*w)
    X = _int_rows(300_000, seed=21) if kind == "int" else _normal_rows(300_000, seed=22)
    b = engine.stage(X)
    p, _ = engine.predict_mlp_proba(m, b)
    labels, _ = engine.predict_mlp(m, b, exact=True)
    mism = np.flatnonzero(p.argmax(axis=1) != labels)
    margin = omlp.logit_margin_f64(X, *w)
    assert mism.size == 0 or margin[mism].max() < 1e-4


def test_drop_in_for_the_quickstart_forward(golden):
    import torch.nn as nn
    import torch.nn.functional as F

    from unionml_b200.predictors import mlp_predict_proba

    class PytorchModel(nn.Module):  # tests/integration/pytorch_app/quickstart.py:14-24
        def __init__(self, in_dims, hidden_dims, out_dims):
            super().__init__()
            self.layers = nn.Sequential(nn.Linear(in_dims, hidden_dims), nn.ReLU(), nn.Linear(hidden_dims, out_dims))

        def forward(self, features):
            return F.softmax(self.layers(features), dim=1)

    torch.manual_seed(0)
    module = PytorchModel(64, 32, 10)
    np.testing.assert_array_equal(module.layers[0].weight.detach().numpy(), golden["w1"])
    frame = pd.DataFrame(np.random.default_rng(4).integers(0, 17, size=(20_000, 64)).astype(np.float64))
    got = mlp_predict_proba(module, frame)
    assert got.dtype == np.float32 and got.shape == (20_000, 10)
    X = frame.values.astype(np.float32)
    with torch.no_grad():
        want = module(torch.from_numpy(frame.values).float()).numpy()
    ref = proba_f64(X, *_weights(golden))
    tol = max(4.0 * float(np.abs(want - ref).max()), 1e-6)
    assert float(np.abs(got - ref).max()) <= tol
    assert float(np.abs(got - want).max()) <= 2 * tol


def test_device_output_and_repeatability(engine, golden):
    w = _weights(golden)
    m = engine.load_mlp(*w)
    X = _int_rows(100_003, seed=31)
    b = engine.stage(X)
    host, _ = engine.predict_mlp_proba(m, b)
    again, _ = engine.predict_mlp_proba(m, b)
    assert np.array_equal(host.view(np.uint32), again.view(np.uint32))
    out = torch.full((100_003 * 10 + 4,), -1.0, dtype=torch.float32, device="cuda")
    none, st = engine.predict_mlp_proba(m, b, out_device_ptr=out.data_ptr())
    assert none is None and st["path"] == 5 and st["d2h_bytes"] == 0
    dev = out[: 100_003 * 10].cpu().numpy().reshape(100_003, 10)
    assert np.array_equal(dev.view(np.uint32), host.view(np.uint32))
    assert (out[100_003 * 10 :].cpu().numpy() == -1.0).all()
    from unionml_b200 import _native as N
    from unionml_b200.engine import EngineError

    with pytest.raises(EngineError) as ei:
        engine.predict_mlp_proba(m, b, out_device_ptr=out.data_ptr() + 4)
    assert ei.value.status == N.UML_ERR_UNSUPPORTED


@pytest.mark.parametrize("force_tc", ["1", "0"])
def test_errors(engine, golden, force_tc, monkeypatch):
    import torch.nn as nn

    from unionml_b200.predictors import mlp_argmax, mlp_predict_proba

    w = _weights(golden)
    module = nn.Sequential(nn.Linear(64, 32), nn.ReLU(), nn.Linear(32, 10))
    with torch.no_grad():
        for layer, (wt, bias) in ((module[0], w[:2]), (module[2], w[2:])):
            layer.weight.copy_(torch.from_numpy(wt))
            layer.bias.copy_(torch.from_numpy(bias))
    for bad in (np.empty((0, 64), dtype=np.float32), np.ones((4, 63), dtype=np.float32)):
        with pytest.raises(ValueError) as want:
            mlp_argmax(module, bad)
        with pytest.raises(ValueError) as got:
            mlp_predict_proba(module, bad)
        assert str(got.value) == str(want.value)
    # NaN / Inf in wrapped device rows, which no staging pass has checked: both fast kernels flag them
    monkeypatch.setenv("UML_B200_MLP_TC", force_tc)
    m = engine.load_mlp(*w)
    for v in (np.nan, np.inf):
        rows = torch.from_numpy(_int_rows(5_000, seed=41)).cuda()
        rows[4_321, 7] = v
        b = engine.wrap_device(rows.data_ptr(), 5_000, 64, keepalive=rows)
        with pytest.raises(ValueError, match="NaN or infinity"):
            engine.predict_mlp_proba(m, b)


def test_full_size_ten_million(engine, golden):
    w = _weights(golden)
    m = engine.load_mlp(*w)
    N = 10_000_000
    X = engine.pinned_empty((N, 64), np.float32)
    for k in range(10):
        X[k * 1_000_000 : (k + 1) * 1_000_000] = np.random.default_rng(k).integers(0, 17, size=(1_000_000, 64), dtype=np.uint8)
    b = engine.stage(X)
    p, st = engine.predict_mlp_proba(m, b)
    assert st["path"] == 5 and st["n_rows"] == N and p.shape == (N, 10)
    assert float(np.abs(p.sum(axis=1, dtype=np.float64) - 1.0).max()) <= 1e-6
    sample = np.random.default_rng(99).choice(N, size=500_000, replace=False)
    assert_within_criterion(p[sample], X[sample], w)
    print(f"mlp proba tcgen05 10M x 64: kernel {st['kernel_ms']:.3f} ms, fp64 {st['recheck_ms']:.3f} ms, flagged {st['n_flagged']}")
