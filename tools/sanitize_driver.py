"""Small-size pass over every shipped kernel, meant to run under compute-sanitizer (see tools/sanitize.sh)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from unionml_b200.engine import Engine  # noqa: E402

z = np.load("tests/golden/digits_lr.npz")
g = np.load("tests/golden/mlp_64_32_10.npz")
eng = Engine(0)
m = eng.load_linear(z["coef"], z["intercept"])
mlp = eng.load_mlp(g["w1"], g["b1"], g["w2"], g["b2"])
X = np.random.default_rng(0).integers(0, 17, size=(40_001, 64), dtype=np.uint8).astype(np.float32)
b = eng.stage(np.asfortranarray(X.astype(np.float64)))  # feature-major float64 source -> transpose kernel
for exact in (True, False):
    eng.predict(m, b, exact=exact)
    eng.predict_mlp(mlp, b, exact=exact)
eng.predict_host(m, X, exact=True, chunk_rows=4096)
buf = eng.device_alloc(b.n_rows)
eng.predict_peers(m, b, [buf.ptr], 0, exact=True, want_stats=True, label_bytes=1)
eng.take_labels(buf.ptr, b.n_rows, np.arange(10.0), label_bytes=1)
# round 2: tensor-core MLP kernel (+ peer stores, queue re-score variant), CUDA-core MLP kernel on float rows, re-score from
# the caller's float64 values, online small-batch kernel, predict_proba, MLP host pipeline, asynchronous host call
import os as _os

eng.predict_mlp_peers(mlp, b, [buf.ptr], 0, exact=True, want_stats=True, label_bytes=1)
Xf = np.random.default_rng(1).standard_normal((20_001, 64))
bf = eng.stage(Xf)
eng.predict_mlp(mlp, bf, exact=True)                     # general floats: FFMA kernel
eng.predict_host(m, Xf, exact=True, chunk_rows=4096)     # float64 source: re-score reads the raw chunk
eng.predict_host(m, np.asfortranarray(Xf[:32]), exact=True)   # online shape: zero-copy kernel, graph replay
eng.predict_host(m, np.asfortranarray(Xf[:32]), exact=True)
eng.predict_proba(m, b)
eng.predict_mlp_host(mlp, X.astype(np.float64), chunk_rows=4096)
eng.predict_host_list(m, X.astype(np.float64), [float(c) for c in range(10)], chunk_rows=4096, asynchronous=True)
m0 = eng.load_linear(np.zeros((5, 64)), np.zeros(5))    # every row a tie: the queue backs up, scoring warps re-score their own rows
eng.predict(m0, b, exact=True)
# fp64 re-score with the feature-major weight table: two rounds of classes (C = 20 -> generic all-rows kernel), an odd
# class count behind the tile kernel, and a wide model whose table is staged in shared memory (F = 784)
rng = np.random.default_rng(4)
m20 = eng.load_linear(rng.standard_normal((20, 64)), rng.standard_normal(20))
eng.predict(m20, b, exact=True)
m3 = eng.load_linear(rng.standard_normal((3, 64)), rng.standard_normal(3))
eng.predict(m3, bf, exact=True)
X784 = (rng.integers(0, 256, size=(6_001, 784)) / 255.0)
m784 = eng.load_linear(rng.standard_normal((10, 784)) * 0.05, rng.standard_normal(10))
eng.predict(m784, eng.stage(X784), exact=True)
eng.predict_host(m784, X784, exact=True, chunk_rows=2048)
# MLP class probabilities: softmax epilogues of the tensor-core kernel (tf32 rows) and the CUDA-core kernel (float rows),
# the fp64 kernel over the flagged rows (rows that are not tf32 values, forced onto the tensor cores) and over all rows
eng.predict_mlp_proba(mlp, b)
eng.predict_mlp_proba(mlp, bf)
_os.environ["UML_B200_MLP_TC"] = "1"
eng.predict_mlp_proba(mlp, bf)
del _os.environ["UML_B200_MLP_TC"]
m48 = eng.load_mlp(rng.standard_normal((48, 64)).astype(np.float32), np.zeros(48, np.float32),
                   rng.standard_normal((10, 48)).astype(np.float32), np.zeros(10, np.float32))
eng.predict_mlp_proba(m48, b)
print("sanitizer driver ok")
