"""MLP class probabilities (uml_mlp_predict_proba) on a resident batch, next to the argmax call on the same rows.

Rows: 10M x 64 cfg-5 inputs (integers 0..16, seeded; tf32 values -> tensor-core kernel, stats path 5) and the same
number of standard-normal rows (CUDA-core kernel, path 3), generated on the device.  Per path: warm-up of at least
0.25 s, then K synchronous calls writing into device memory; the engine's CUDA events give the scoring kernel's time
(kernel_ms) and the fp64 kernel's behind it (recheck_ms).  Traffic model: 4 F bytes read + 4 C bytes written per row
(296 B at 64 -> 32 -> 10) against the 6 489.6 GB/s device-to-device copy peak measured for this project.  A 200 000-row
sample of each output is checked against the float64 softmax before anything is reported.

    python tools/bench_mlp_proba.py --steps 50 --out profiles/r03_mlp_proba.json
    python tools/bench_mlp_proba.py --ab-store 3 ...   # same-box A/B of the two store schemes, alternating processes
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

COPY_PEAK_GBS = 6489.6


def device_facts() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return {"device": name, "power_limit_w": float(power), "max_sm_mhz": float(clk)}
    except Exception as exc:  # noqa: BLE001 - still report what torch knows
        import torch

        return {"device": torch.cuda.get_device_name(0), "power_limit_w": None, "max_sm_mhz": None,
                "nvidia_smi": f"unavailable: {exc}"}


def proba_f64(X, w1, b1, w2, b2):
    from oracle import mlp as omlp

    z = omlp.logits(X, w1, b1, w2, b2, np.float64)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return e / e.sum(axis=1, keepdims=True)


def check_sample(p_dev, X_dev, w, n=200_000) -> dict:
    """max |p - p_f64| on a row sample against max(4 max |p_torch - p_f64|, 1e-6) (tests/test_gpu_mlp_proba.py)."""
    import torch

    idx = torch.from_numpy(np.random.default_rng(7).choice(X_dev.shape[0], size=n, replace=False)).cuda()
    X = X_dev[idx].cpu().numpy()
    p = p_dev[idx].cpu().numpy().astype(np.float64)
    ref = proba_f64(X, *w)
    t = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)) for a in (X, *w)]
    with torch.no_grad():
        pt = torch.softmax(torch.nn.functional.linear(torch.relu(torch.nn.functional.linear(t[0], t[1], t[2])), t[3], t[4]), 1)
    tol = max(4.0 * float(np.abs(pt.numpy() - ref).max()), 1e-6)
    err = float(np.abs(p - ref).max())
    row_sum = float(np.abs(p.sum(axis=1) - 1.0).max())
    if err > tol or row_sum > 1e-6:
        raise SystemExit(f"output check failed: max err {err:.3g} (tolerance {tol:.3g}), row-sum error {row_sum:.3g}")
    return {"rows": n, "max_abs_err": err, "tolerance": tol, "max_row_sum_err": row_sum}


def timed(fn, steps: int, warmup: int) -> dict:
    t_end = time.perf_counter() + 0.25
    w = 0
    while w < warmup or time.perf_counter() < t_end:
        fn()
        w += 1
    kern, rechk, calls = [], [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        st = fn()  # synchronous: returns after the device has finished
        calls.append((time.perf_counter() - t0) * 1e3)
        kern.append(st["kernel_ms"])
        rechk.append(st["recheck_ms"])
    return {"path": st["path"], "n_flagged": st["n_flagged"], "kernel_launches": st["kernel_launches"],
            "kernel_ms": float(np.mean(kern)), "kernel_ms_min": float(np.min(kern)), "recheck_ms": float(np.mean(rechk)),
            "call_ms": float(np.median(calls)), "warmup_calls": w}


def run(args) -> dict:
    import torch

    from unionml_b200.engine import Engine

    g = np.load(ROOT / "tests" / "golden" / "mlp_64_32_10.npz")
    w = (g["w1"], g["b1"], g["w2"], g["b2"])
    F, C = w[0].shape[1], w[2].shape[0]
    N = args.rows
    eng = Engine(0)
    m = eng.load_mlp(*w)
    gen = torch.Generator(device="cuda").manual_seed(5)
    rows = {
        "tf32_int": torch.randint(0, 17, (N, F), generator=gen, device="cuda", dtype=torch.int32).float(),
        "normal": torch.randn((N, F), generator=gen, device="cuda"),
    }
    out = torch.empty((N, C), dtype=torch.float32, device="cuda")
    labels = torch.empty(N, dtype=torch.int32, device="cuda")
    bytes_per_row = 4 * F + 4 * C
    floor_ms = N * bytes_per_row / (COPY_PEAK_GBS * 1e9) * 1e3
    res = {"rows": N, "shape": [F, w[0].shape[0], C], "steps": args.steps, "store": os.environ.get("UML_B200_MLP_PROBA_STORE", "default"),
           "bytes_per_row": bytes_per_row, "copy_peak_gbs": COPY_PEAK_GBS, "roofline_floor_ms": floor_ms, "paths": {}}
    for name, X in rows.items():
        b = eng.wrap_device(X.data_ptr(), N, F, keepalive=X)
        proba = lambda: eng.predict_mlp_proba(m, b, out_device_ptr=out.data_ptr())[1]  # noqa: E731
        argmax = lambda: eng.predict_mlp(m, b, exact=True, out_device_ptr=labels.data_ptr())[1]  # noqa: E731
        argmax_fast = lambda: eng.predict_mlp(m, b, exact=False, out_device_ptr=labels.data_ptr())[1]  # noqa: E731
        proba()
        check = check_sample(out, X, w)
        entry = {"check": check}
        for label, fn in (("proba", proba), ("argmax_exact", argmax), ("argmax_fast", argmax_fast)):
            t = timed(fn, args.steps, args.warmup)
            t["rows_per_s"] = N / (t["kernel_ms"] * 1e-3)
            if label == "proba":
                t["roofline_fraction"] = floor_ms / t["kernel_ms"]
            entry[label] = t
        res["paths"][name] = entry
        print(f"{name}: proba kernel {entry['proba']['kernel_ms']:.3f} ms (path {entry['proba']['path']}, "
              f"{entry['proba']['roofline_fraction']:.2f} of the {bytes_per_row} B/row floor {floor_ms:.3f} ms), "
              f"argmax exact {entry['argmax_exact']['kernel_ms']:.3f} / fast {entry['argmax_fast']['kernel_ms']:.3f} ms",
              flush=True)
        del b
    res.update(device_facts())
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ab-store", type=int, default=0, help="rounds of direct/staged processes (same-box A/B)")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_mlp_proba.json"))
    args = ap.parse_args()
    if args.ab_store:
        rounds = []
        for r in range(args.ab_store):
            for store in ("direct", "staged"):
                env = dict(os.environ, UML_B200_MLP_PROBA_STORE=store)
                tmp = Path(args.out).with_suffix(f".{store}{r}.tmp.json")
                cmd = [sys.executable, __file__, "--rows", str(args.rows), "--steps", str(args.steps),
                       "--warmup", str(args.warmup), "--out", str(tmp)]
                subprocess.run(cmd, env=env, check=True)
                rounds.append(json.loads(tmp.read_text()))
                tmp.unlink()
        summary = {s: {p: [r["paths"][p]["proba"]["kernel_ms"] for r in rounds if r["store"] == s] for p in rounds[0]["paths"]}
                   for s in ("direct", "staged")}
        result = {"ab_store": summary, "rounds": rounds, **device_facts()}
    else:
        result = run(args)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result.get("ab_store", {}), indent=1))


if __name__ == "__main__":
    main()
