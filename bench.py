#!/usr/bin/env python
"""bench.py - rows/sec of the batch-predict hot path on N B200s (BASELINE.json metric, configs[1] by default).

    python bench.py --gpus 1 --steps 20 --warmup 5                      # this repo's CUDA path, cfg 2 (10M x 64 -> 10)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1      # the reference's CPU path, same metric
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                          # one rank per GPU
    ... --config cfg3 | cfg5        # 784 -> 10 logistic on 50M rows / 2-layer MLP 64 -> 32 -> 10 on 10M rows
    ... --scaling weak              # r01 mode: every GPU scores its own 10M rows (default: strong - ONE batch split)
    ... --dump-outputs DIR          # after the timed steps: DIR/labels.npy, the last timed step's labels (see dump_labels)

A "step" is one pass of the hot path over one batch.  At N > 1 the batch is split across the GPUs (north_star: "the
batch is split across GPUs", SURVEY.md 8e partition [r*N/G, (r+1)*N/G)), every rank scores its shard in EXACT mode
and the uint8 label vector is exchanged so every rank holds all labels.

`value`  : whole-job rows/s with the shard resident in HBM (CUDA events on the launching stream, barrier + synchronize
           on both sides, max over ranks).
`e2e`    : the same metric through the reference-facing plugin with HOST buffers: a float64 feature-major pandas
           DataFrame (what Dataset.get_features yields, /root/reference/unionml/dataset.py:506-520) ->
           Model.predict(features=frame) -> List[float]  - the reference arm's own input and output types.  The
           pinned-fp32 -> int32-labels engine call of round 1 is reported beside it (`e2e.engine_pinned_f32`).
`roofline`: algorithmic bytes (4 F per row) / CUDA-event duration of the scoring kernel, against MEASURED_PEAKS.json.
`cpu_baseline`: the reference predictor as written, on this box's host cores, on a bounded sample - the only place,
           with --impl reference, where oracle/ code runs.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the bench writes nothing into the tree it runs from (it may be read-only)

UNIT = "rows/s"
CONFIGS = {
    "cfg2": {
        "metric": "rows/sec batch predict (64->10 logistic)", "kind": "linear", "F": 64, "C": 10, "rows": 10_000_000,
        "data": "digits", "kernel": "linear_argmax_tma_kernel<10, EXACT, QUEUE> (fp64 re-score by a tenth warp of the same launch)", "cpu_rows": 2_000_000,
        "what": "BASELINE.json configs[1]: digits predictor (golden LogisticRegression 64->10)",
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch on 10M rows (profiles/r02_linear_argmax_tma_queue.ncu_raw.csv)
        "traffic_10m": 2_568_923_504, "traffic_src": "profiles/r02_linear_argmax_tma_queue.ncu_raw.csv (ncu --set full, per launch: dram read 2.560358 GB + write 8.565504 MB)",
    },
    "cfg3": {
        "metric": "rows/sec batch predict (784->10 logistic)", "kind": "linear", "F": 784, "C": 10, "rows": 50_000_000,
        "data": "mnist", "kernel": "linear_argmax_tma_kernel<10, EXACT>", "cpu_rows": 300_000,
        "what": "BASELINE.json configs[2]: MNIST-shaped 784->10 logistic (W ~ N(0, 0.05), b ~ N(0, 1), X = uint8 / 255)",
        "traffic_10m": None, "traffic_src": None,
    },
    "cfg5": {
        "metric": "rows/sec batch predict (2-layer MLP 64->32->10)", "kind": "mlp", "F": 64, "C": 10, "rows": 10_000_000,
        "data": "digits", "kernel": "mlp_argmax_tc_kernel<32, 10, EXACT> (tcgen05 kind::tf32)", "cpu_rows": 200_000,
        "what": "BASELINE.json configs[4]: PyTorch 2-layer MLP predictor (torch.manual_seed(0) PytorchModel(64, 32, 10))",
        "traffic_10m": 2_568_177_568, "traffic_src": "profiles/r02_mlp_argmax_tc.ncu_raw.csv (ncu --set full, per launch: dram read 2.560164 GB + write 8.013568 MB)",
    },
}
CHUNK = 1_000_000  # digits rows are generated in global 1M-row chunks: chunk k = default_rng(k)
DUMP_ALL_ROWS = 12_000_000  # --dump-outputs writes every label up to this many rows (48 MB of float32) ...
DUMP_SAMPLE_ROWS = 4_000_000  # ... and a seeded sample of this many rows (+ their indices, 48 MB in all) above it


# ---------------------------------------------------------------------------------------------------------------
# data and models (deterministic; SURVEY.md 8d)
# ---------------------------------------------------------------------------------------------------------------
def digits_rows(lo: int, hi: int, out: np.ndarray) -> None:
    """Global rows [lo, hi) of the cfg-2 batch into `out`: chunk k = default_rng(k).integers(0, 17, (1M, 64), uint8)."""
    for k in range(lo // CHUNK, (hi + CHUNK - 1) // CHUNK):
        c0, c1 = k * CHUNK, (k + 1) * CHUNK
        a, b = max(lo, c0), min(hi, c1)
        if a >= b:
            continue
        chunk = np.random.default_rng(k).integers(0, 17, size=(CHUNK, 64), dtype=np.uint8)
        out[a - lo : b - lo] = chunk[a - c0 : b - c0]


def mnist_rows_device(torch, dev, seed_rank: int, rows: int, F: int = 784):
    """cfg-3 shard generated ON the device: uint8 pixels / 255 in fp32, generator seeded per shard (SURVEY.md 8d)."""
    g = torch.Generator(device=dev).manual_seed(1000 + seed_rank)
    X = torch.empty((rows, F), dtype=torch.float32, device=dev)
    for r0 in range(0, rows, CHUNK):
        n = min(CHUNK, rows - r0)
        X[r0 : r0 + n] = torch.randint(0, 256, (n, F), generator=g, device=dev, dtype=torch.uint8).to(torch.float32) / 255.0
    return X


def load_model_arrays(cfg):
    if cfg["kind"] == "mlp":
        z = np.load(ROOT / "tests" / "golden" / "mlp_64_32_10.npz")
        return {"w1": z["w1"], "b1": z["b1"], "w2": z["w2"], "b2": z["b2"]}
    if cfg["data"] == "mnist":
        return {"coef": (np.random.default_rng(1).standard_normal((10, 784)) * 0.05).astype(np.float32),
                "intercept": np.random.default_rng(2).standard_normal(10).astype(np.float32), "classes": np.arange(10)}
    z = np.load(ROOT / "tests" / "golden" / "digits_lr.npz")
    return {"coef": z["coef"], "intercept": z["intercept"], "classes": z["classes"]}


def sklearn_estimator(arrs, F):
    from sklearn.linear_model import LogisticRegression

    est = LogisticRegression(C=1.0, max_iter=1000)
    est.coef_, est.intercept_, est.classes_, est.n_features_in_ = arrs["coef"], arrs["intercept"], arrs["classes"], F
    return est


def torch_module(arrs):
    import torch
    import torch.nn as nn
    import torch.nn.functional as Fn

    class PytorchModel(nn.Module):  # /root/reference/tests/integration/pytorch_app/quickstart.py:14-24
        def __init__(self, in_dims, hidden_dims, out_dims):
            super().__init__()
            self.layers = nn.Sequential(nn.Linear(in_dims, hidden_dims), nn.ReLU(), nn.Linear(hidden_dims, out_dims))

        def forward(self, features):
            return Fn.softmax(self.layers(features), dim=1)

    m = PytorchModel(arrs["w1"].shape[1], arrs["w1"].shape[0], arrs["w2"].shape[0])
    with torch.no_grad():
        m.layers[0].weight.copy_(torch.from_numpy(arrs["w1"]))
        m.layers[0].bias.copy_(torch.from_numpy(arrs["b1"]))
        m.layers[2].weight.copy_(torch.from_numpy(arrs["w2"]))
        m.layers[2].bias.copy_(torch.from_numpy(arrs["b2"]))
    return m.eval()


def float64_labels(cfg, arrs, X64: np.ndarray) -> np.ndarray:
    """Class index per row in float64 numpy (inline check of the bench, not the oracle package)."""
    if cfg["kind"] == "mlp":
        h = np.maximum(X64 @ arrs["w1"].astype(np.float64).T + arrs["b1"].astype(np.float64), 0.0)
        return (h @ arrs["w2"].astype(np.float64).T + arrs["b2"].astype(np.float64)).argmax(1)
    return (X64 @ arrs["coef"].astype(np.float64).T + arrs["intercept"].astype(np.float64)).argmax(1)


def dump_labels(out_dir: str, labels: np.ndarray) -> None:
    """--dump-outputs: DIR/labels.npy, the class index of every row of the global batch as float32.

    Above DUMP_ALL_ROWS rows it holds a fixed sample instead (DUMP_SAMPLE_ROWS rows drawn by default_rng(0), in row
    order) and DIR/rows.npy the global row index of each entry (float64).  The inputs are seeded, so two builds run with
    the same arguments can be compared label for label."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    if labels.shape[0] > DUMP_ALL_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(labels.shape[0], DUMP_SAMPLE_ROWS, replace=False))
        labels = labels[rows]
        np.save(out / "rows.npy", rows.astype(np.float64))
    else:
        (out / "rows.npy").unlink(missing_ok=True)
    np.save(out / "labels.npy", labels.astype(np.float32))


def measured_peak_hbm():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def usable_cores() -> int:
    """Host threads this process may really run: min(affinity, cgroup cpu quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = (
        "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
        "clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
# CPU legs (the only users of oracle/)
# ---------------------------------------------------------------------------------------------------------------
def lift_thread_limits():
    """torchrun exports OMP_NUM_THREADS=1; the reference arm must use the host cores it can (VERDICT r1 weak #9)."""
    n = usable_cores()
    try:  # load every threaded library first: the limits only reach pools that exist when they are set
        import pandas  # noqa: F401
        import sklearn.linear_model  # noqa: F401
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=n)
    except Exception:
        pass
    try:
        import torch

        torch.set_num_threads(n)
    except Exception:
        pass
    return n


def blas_threads() -> int:
    try:
        from threadpoolctl import threadpool_info

        return max([i.get("num_threads", 1) for i in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_sample_frame(cfg, sample_rows: int):
    import pandas as pd

    F = cfg["F"]
    if cfg["data"] == "mnist":
        X = np.random.default_rng(7).integers(0, 256, size=(sample_rows, F)).astype(np.float64) / 255.0
    else:
        X32 = np.empty((sample_rows, F), dtype=np.float32)
        digits_rows(0, sample_rows, X32)
        X = X32.astype(np.float64)
    return pd.DataFrame(X, columns=[f"pixel_{i}" for i in range(F)])


def cpu_reference_predict_rows_per_s(cfg, arrs, sample_rows: int, repeats: int):
    """The reference's CPU path on host cores: Model.predict(features=frame) -> the canonical predictor as written.

    Restated wrapper (oracle.unionml_path, no flytekit) + the real library arithmetic (scikit-learn / torch), float64
    frame as the reference's DataFrame path feeds it.  Returns (rows/s best-of-repeats, seconds list)."""
    import pandas as pd

    from oracle import unionml_path as opath

    frame = cpu_sample_frame(cfg, sample_rows)

    def reader() -> pd.DataFrame:
        return frame

    if cfg["kind"] == "mlp":
        import torch

        module = torch_module(arrs)

        def predictor(model, features) -> list:  # quickstart.py:68-70 (+ process_features :31-32)
            return [float(x) for x in model(torch.from_numpy(features.values).float()).argmax(1)]

        model_object = module
    else:
        est = sklearn_estimator(arrs, cfg["F"])
        est.feature_names_in_ = np.asarray(frame.columns, dtype=object)

        def predictor(estimator, features) -> list:  # /root/reference/README.md:87-92
            return [float(x) for x in estimator.predict(features)]

        model_object = est
    spec = opath.PathSpec(reader=reader, targets=["target"], predictor=predictor, model_object=model_object)
    times = []
    out = None
    for _ in range(repeats):
        out = None  # the previous step's list is released outside the timed region (both arms do this)
        t0 = time.perf_counter()
        out = opath.predict(spec, features=frame)
        times.append(time.perf_counter() - t0)
        assert len(out) == sample_rows
    return sample_rows / min(times), times


def cpu_sample_note(cfg, sample, cores):
    lib = "torch CPU PytorchModel forward + [float(x) for x in ...argmax(1)]" if cfg["kind"] == "mlp" else \
        "scikit-learn LogisticRegression.predict + [float(x) ...]"
    return (f"{sample} rows/step of the {cfg['what'].split(':')[0]} batch as a float64 DataFrame through the restated "
            f"Model.predict(features=...) wrapper + {lib} (BLAS threads={cores}, usable cores={usable_cores()}, "
            f"os.cpu_count()={os.cpu_count()})")


def run_reference_arm(args, cfg):
    """--impl reference: same metric/unit/config, CPU only; under torchrun only rank 0 works."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    lift_thread_limits()
    arrs = load_model_arrays(cfg)
    sample = args.cpu_rows or cfg["cpu_rows"]
    for _ in range(max(args.warmup, 1)):
        cpu_reference_predict_rows_per_s(cfg, arrs, min(sample, 100_000), 1)
    per_step = []
    for _ in range(args.steps):
        _, times = cpu_reference_predict_rows_per_s(cfg, arrs, sample, 1)
        per_step.append(times[0])
    value = sample / statistics.mean(per_step)
    cores = blas_threads()
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(per_step),
        "higher_is_better": True, "scaling": args.scaling_resolved, "vs_baseline": None, "dtype": "f64" if cfg["kind"] == "linear" else "f32",
        "data": "synthetic",
        "config": workload_config(args, cfg, args.gpus) | {"sample_rows_per_step": sample,
                                                         "note": "CPU time is linear in rows: each step times a bounded sample of the workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": cpu_sample_note(cfg, sample, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def global_rows(args, cfg, n_gpus: int) -> int:
    if args.rows:
        return args.rows * (n_gpus if args.scaling_resolved == "weak" else 1)
    if args.scaling_resolved == "weak":
        return cfg["rows"] * n_gpus if cfg["data"] != "mnist" else 6_250_000 * n_gpus
    if cfg["data"] == "mnist" and n_gpus < 4:
        # 50M x 784 fp32 is 156.8 GB: it needs >= 4 GPUs; below that the bench scores the 8-GPU shard size per GPU
        return 6_250_000 * n_gpus
    return cfg["rows"]


def workload_config(args, cfg, n_gpus: int) -> dict:
    g = global_rows(args, cfg, n_gpus)
    F = cfg["F"]
    return {
        "workload": f"{cfg['what']}, {g} x {F} synthetic fp32 rows "
        + ("(integers 0..16)" if cfg["data"] == "digits" else "(uint8 / 255, generated on the device per shard)"),
        "config": args.config, "global_rows": g, "rows_per_gpu": g // max(n_gpus, 1), "n_features": F, "n_classes": cfg["C"],
        "mode": "exact (fp32 / tf32x2-split scores + margin guard + fp64 re-score; labels == the float64 argmax)",
        "labels": "uint8 class index per row",
        "parallelism": (f"row-sharded x{n_gpus} ({args.scaling_resolved} scaling), label exchange: " + getattr(args, "gather_used", args.gather))
        if n_gpus > 1 else "single GPU",
        "l2_policy": f"inputs ({g // max(n_gpus, 1) * 4 * F / 1e9:.2f} GB/step/GPU) are larger than L2 (126 MB); no flush needed",
    }


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def run_gpu_arm(args, cfg):
    import pandas as pd
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from unionml_b200.engine import Engine
    from unionml_b200.sharding import PeerLabelExchange, predict_sharded, shard_bounds, shard_counts

    eng = Engine(local_rank)
    # an explicit (non-default) torch stream is both torch's current stream and the engine's launch stream, so the
    # torch.cuda.Event pair below brackets exactly the library's kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)

    F, kind = cfg["F"], cfg["kind"]
    arrs = load_model_arrays(cfg)
    model = eng.load_mlp(arrs["w1"], arrs["b1"], arrs["w2"], arrs["b2"]) if kind == "mlp" else \
        eng.load_linear(arrs["coef"], arrs["intercept"], arrs["classes"])
    G = global_rows(args, cfg, world)
    lo, hi = shard_bounds(G, rank, world)
    rows = hi - lo
    counts = shard_counts(G, world)

    # ---- this rank's shard, resident in HBM ----
    X_host = None
    if cfg["data"] == "digits":
        X_host = eng.pinned_empty((rows, F), np.float32)  # also the source of the engine-level e2e leg
        digits_rows(lo, hi, X_host)
        batch = eng.stage(X_host)
    else:
        X_dev = mnist_rows_device(torch, dev, rank, rows, F)
        batch = eng.wrap_device(X_dev.data_ptr(), rows, F, F, keepalive=X_dev)

    def predict_into(ptrs, row_offset, want_stats=False, b=None):
        fn = eng.predict_mlp_peers if kind == "mlp" else eng.predict_peers
        return fn(model, b or batch, ptrs, row_offset, exact=True, want_stats=want_stats, label_bytes=1)

    # ---- label exchange back-ends (N > 1): fused epilogue stores / local store + copy kernel / pipelined / NCCL ----
    candidates = {}
    if world > 1:
        wanted = ["fused", "push", "push4", "nccl"] if args.gather == "auto" else [args.gather]
        for name in wanted:
            if name == "nccl":
                candidates[name] = None
                continue
            try:
                candidates[name] = PeerLabelExchange(G, dev, dtype=torch.uint8, multicast=not args.no_multicast,
                                                     push=name.startswith("push"), pipeline=4 if name == "push4" else 1)
            except Exception as exc:  # symmetric memory unavailable on this box
                if rank == 0:
                    print(f"bench: {name}: symmetric memory unavailable ({exc!r})", file=sys.stderr)
        if not candidates:
            candidates["nccl"] = None
    labels_plain = torch.empty(G, dtype=torch.uint8, device=dev)  # N = 1 vector / NCCL target

    def make_step(name):
        ex = candidates.get(name) if world > 1 else None
        if world == 1:
            return lambda: predict_into([labels_plain.data_ptr()], 0), labels_plain
        if ex is not None:
            return (lambda: predict_sharded(eng, model, batch, row_offset=lo, counts=counts, exact=True, exchange=ex)), ex.labels

        def nccl_step():
            predict_into([labels_plain.data_ptr()], lo)
            if len(set(counts)) == 1:
                dist.all_gather_into_tensor(labels_plain, labels_plain[lo:hi])
            else:
                from unionml_b200.sharding import gather_labels

                labels_plain.copy_(gather_labels(labels_plain[lo:hi].clone(), counts))
        return nccl_step, labels_plain

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(step, k):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for i in range(k):
            step()
            # bound the number of queued cross-rank barrier steps (a 1250-deep untimed queue did not drain at N = 2)
            if world > 1 and (i + 1) % 64 == 0 and i + 1 < k:
                torch.cuda.synchronize()
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / k

    # ---- pick the exchange (N > 1, --gather auto): a short A/B of the back-ends in this process, same data ----
    gather_ab = {}
    chosen = "none"
    if world > 1:
        for name in candidates:
            step, _ = make_step(name)
            for _ in range(3):
                step()
            gather_ab[name] = timed_steps(step, 10)
        chosen = min(gather_ab, key=gather_ab.get)
    step, labels_all = make_step(chosen)
    ex = candidates.get(chosen) if world > 1 else None
    # N > 1: a step is 2-4 launches of 60-200 us in total, issued from Python on every rank; capture it once in a CUDA
    # graph and replay it, so the timed loop measures the GPUs and not the launch rate of the host.  Falls back to
    # eager launches when the capture is refused (reported in the JSON line).
    graph_note = "eager launches"
    if world > 1 and not args.no_graph:
        eager_step = step
        try:
            for _ in range(3):
                eager_step()
            barrier()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                eager_step()
            barrier()
            g.replay()
            barrier()
            step = g.replay
            graph_note = "one CUDA graph per step (captured once, replayed)"
        except Exception as exc:  # capture refused: keep launching eagerly
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
            torch.cuda.set_stream(stream)
            eng.set_stream(stream.cuda_stream)
            step = eager_step
            graph_note = f"eager launches (graph capture failed: {type(exc).__name__})"
        # every rank must take the same route
        flag = torch.tensor([1 if step is not eager_step else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and step is not eager_step:
            step = eager_step
            graph_note = "eager launches (a peer rank could not capture)"
    how = "one NVLS multicast store per tile" if (ex is not None and ex.multicast) else "one store per peer per tile"
    args.gather_used = {
        "fused": f"fused uint8 label stores ({how}) from the kernel epilogue over NVLink (symmetric memory) + barrier",
        "push": f"kernel stores uint8 labels locally, thin copy kernel pushes the slice ({how.replace(' per tile', '')}) + barrier",
        "push4": "shard scored as 4 sub-batches; a copy kernel on a side stream pushes sub-batch j's labels "
                 f"({how.replace(' per tile', '')}) under the scoring kernel of sub-batch j+1, + barrier",
        "nccl": "ncclAllGather of uint8 labels", "none": "none"}[chosen]

    # warm-up: at least W steps, and keep going until the GPU has been under this load for ~0.25 s - the shard was just
    # generated on the host for seconds, the clocks are at idle, and K x 0.4 ms of timed region would otherwise sit on
    # the boost ramp (same-box A/B: 0.373 ms/step warm vs 0.40 right after idle)
    n_warm = 0
    if world == 1:
        t_warm = time.perf_counter()
        while n_warm < max(args.warmup, 3) or (time.perf_counter() - t_warm < 0.25 and n_warm < 4000):
            step()
            n_warm += 1
            if n_warm % 32 == 0:
                torch.cuda.synchronize()
    else:  # every rank must run the same number of (barrier-carrying) steps: derive it from the all-reduced A/B time
        n_target = max(args.warmup, 3, min(4000, int(250.0 / max(gather_ab[chosen], 0.02))))
        while n_warm < n_target:
            step()
            n_warm += 1
            if n_warm % 32 == 0:
                torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- timed region: exactly K steps, CUDA events on the launching stream ----
    ms_per_step = timed_steps(step, args.steps)
    value = G / (ms_per_step * 1e-3)
    # the labels the last timed step left, copied out before the untimed steps below write the vector again
    dumped = labels_all.cpu().numpy() if args.dump_outputs and rank == 0 else None

    # ---- roofline of the dominant kernel: CUDA events around the scoring kernel inside the library, live ----
    k_ms, r_ms, flagged, launches_per_step, path = [], [], 0, 2, 0
    for _ in range(args.steps):
        if ex is not None and not ex.push:
            st = predict_into(ex.peer_ptrs, lo, want_stats=True)  # the variant the step really runs
            ex.barrier()
        else:
            tgt = ex.own_ptr if ex is not None else labels_plain.data_ptr()
            st = predict_into([tgt], lo if world > 1 else 0, want_stats=True)
        k_ms.append(st["kernel_ms"])
        r_ms.append(st["recheck_ms"])
        flagged, launches_per_step, path = st["n_flagged"], st["kernel_launches"], st["path"]
    # this repo's kernels per step: the scoring launches the library reports, plus its label-push copy kernel where the
    # exchange uses one (push: 1; push4: 4 sub-batches, each scored and pushed); torch's barrier / NCCL are not counted
    if chosen == "push":
        launches_per_step += 1
    elif chosen == "push4":
        launches_per_step = 4 * (launches_per_step + 1)
    kernel_ms = statistics.mean(k_ms)
    if kind == "mlp" and path != 5:
        raise SystemExit(f"bench: cfg5 must run the tensor-core kernel (stats path 5), got path {path}")
    # keep the same load running (untimed) until nvidia-smi has had ~0.6 s to sample clocks under it (N = 1 only)
    if world == 1:
        for _ in range(min(5000, int(600.0 / max(ms_per_step, 0.05)))):
            step()
        torch.cuda.synchronize()
    exchange_ms = None
    if world > 1:  # cost of the label exchange alone, CUDA events, same stream
        def exchange_only():
            if ex is not None:
                if ex.push:
                    off = lo
                    remote = ex.peer_ptrs if ex.multicast else ex.peer_ptrs[1:]
                    eng.push_labels(ex.own_ptr + off, [p + off for p in remote], rows)
                ex.barrier()
            elif len(set(counts)) == 1:
                dist.all_gather_into_tensor(labels_plain, labels_plain[lo:hi])
        exchange_ms = timed_steps(exchange_only, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    peak, peak_src = measured_peak_hbm()
    bytes_per_launch = rows * 4 * F
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    traffic = args.traffic if args.traffic is not None else (cfg["traffic_10m"] if rows == 10_000_000 else None)
    roofline = {
        "bound": "hbm", "kernel": cfg["kernel"], "achieved": achieved, "peak": peak, "peak_source": peak_src,
        "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": cfg["traffic_src"] if traffic else None,
        "kernel_ms": kernel_ms, "kernel_ms_min": min(k_ms), "rescore_ms": statistics.mean(r_ms), "exchange_ms": exchange_ms,
        "algorithmic_bytes_per_launch": bytes_per_launch, "rows_per_launch": rows, "rows_rescored_fp64": flagged,
        "note": "per-GPU kernel (this rank's shard); at N > 1 the launch covers global_rows / N rows",
    }

    # ---- parity inside the bench: device labels vs float64 numpy on a sample of EVERY rank's rows ----
    step()
    torch.cuda.synchronize()
    sample_n = min(args.check_rows, min(counts))
    if cfg["data"] == "digits":
        for r in range(world if rank == 0 else 0):
            rlo, _ = shard_bounds(G, r, world)
            Xs = np.empty((sample_n, F), dtype=np.float32)
            digits_rows(rlo, rlo + sample_n, Xs)
            want = float64_labels(cfg, arrs, Xs.astype(np.float64))
            got = labels_all[rlo : rlo + sample_n].cpu().numpy()
            if not np.array_equal(got.astype(np.int64), want):
                raise SystemExit(f"bench: labels of rank {r}'s first {sample_n} rows differ from float64 numpy (as seen on rank 0)")
    else:  # device-generated shard: every rank checks its own first rows against float64 numpy, streamed
        Xs = X_dev[:sample_n].cpu().numpy().astype(np.float64)
        want = float64_labels(cfg, arrs, Xs)
        got = labels_all[lo : lo + sample_n].cpu().numpy()
        ok = torch.tensor([int(np.array_equal(got.astype(np.int64), want))], device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) != 1:
            raise SystemExit("bench: labels differ from float64 numpy on the checked rows of some rank")
    if world > 1:
        # every rank must hold every rank's labels: compare the exchanged vector with a plain NCCL all-gather
        mine = labels_all[lo:hi].clone()
        from unionml_b200.sharding import gather_labels

        ref_all = gather_labels(mine, counts)
        torch.cuda.synchronize()
        if not torch.equal(ref_all, labels_all):
            raise SystemExit(f"bench: rank {rank}: exchanged label vector differs from the NCCL all-gather")

    # ---- e2e legs: HOST buffers in, HOST results out, copies inside the timed region ----
    e2e = run_e2e_legs(args, cfg, arrs, eng, model, torch, dist, dev, rank, world, lo, hi, X_host, X_dev if cfg["data"] != "digits" else None,
                       labels_all, barrier, pd)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        lift_thread_limits()  # the CPUs this container may really use (cgroup quota), not os.cpu_count() threads
        sample = args.cpu_rows or cfg["cpu_rows"]
        rps, times = cpu_reference_predict_rows_per_s(cfg, arrs, sample, 3)
        cores = blas_threads()
        extra = {}
        if kind == "linear" and cfg["data"] == "digits":
            est_nd = sklearn_estimator(arrs, F)
            Xnd = X_host[:sample].astype(np.float64)
            nd_t = []
            for _ in range(3):
                t0 = time.perf_counter()
                est_nd.predict(Xnd)
                nd_t.append(time.perf_counter() - t0)
            extra["ndarray_value"] = sample / min(nd_t)
            extra["ndarray_note"] = "bare LogisticRegression.predict on a C-order float64 ndarray (no DataFrame, no list conversion)"
            try:  # plain-C OpenMP restatement (oracle/linear_predict.c): what the host cores can do without Python in the way
                from oracle import c_port

                rows_c = X_host[:sample]
                c_port.predict_indices(rows_c[:10_000], arrs["coef"], arrs["intercept"])
                ct = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    idx_c = c_port.predict_indices(rows_c, arrs["coef"], arrs["intercept"])
                    ct.append(time.perf_counter() - t0)
                extra.update({"c_port_value": sample / min(ct), "c_port_threads": c_port.num_threads(),
                              "c_port_note": "oracle/linear_predict.c, float64 scores over the fp32 rows, OpenMP over rows; labels "
                              + ("equal" if np.array_equal(idx_c, labels_all[:sample].cpu().numpy()) else "DIFFER from") + " the GPU's"})
            except Exception as exc:  # the C port is optional evidence, never a reason to lose the bench line
                extra.update({"c_port_value": None, "c_port_note": f"unavailable: {exc!r}"})
        cpu_baseline = {**extra, "value": rps, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": cpu_sample_note(cfg, sample, cores) + ", best of 3"}

    if dumped is not None:
        dump_labels(args.dump_outputs, dumped)
    if rank == 0:
        line = {
            "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling_resolved, "vs_baseline": None, "dtype": "f32" if kind == "linear" else "tf32x2+f32",
            "data": "synthetic", "config": workload_config(args, cfg, world), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "e2e": e2e, "clocks": clocks, "gpu_launches": launches_per_step * args.steps,
            "gather_ab_ms_per_step": gather_ab or None, "step_launch": graph_note if world > 1 else "eager launches",
            "device": eng.info,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_e2e_legs(args, cfg, arrs, eng, model, torch, dist, dev, rank, world, lo, hi, X_host, X_dev, labels_all, barrier, pd):
    """(1) the plugin boundary: float64 feature-major DataFrame -> Model.predict(features=frame) -> List[float];
    (2) the engine call: pinned fp32 rows -> int32 labels.  Per-rank shard (cfg 3: a bounded 1M-row host sample of
    the shard - 156.8 GB of rows do not fit in host memory), wall clock, max over ranks."""
    from typing import List

    from unionml_b200 import Dataset, Model
    from unionml_b200.predictors import linear_argmax, mlp_argmax

    F, kind = cfg["F"], cfg["kind"]
    rows = hi - lo
    if args.skip_e2e:
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "--skip-e2e (profiling run)"}
    e2e_rows = rows if cfg["data"] == "digits" else min(rows, 1_000_000)
    # feature-major float64 block, exactly what a pandas frame of the features holds (SURVEY.md hard part 6)
    Xfm = np.empty((F, e2e_rows), dtype=np.float64)
    if cfg["data"] == "digits":
        for r0 in range(0, e2e_rows, CHUNK):
            r1 = min(e2e_rows, r0 + CHUNK)
            Xfm[:, r0:r1] = X_host[r0:r1].T
    else:
        for r0 in range(0, e2e_rows, 250_000):
            r1 = min(e2e_rows, r0 + 250_000)
            Xfm[:, r0:r1] = X_dev[r0:r1].cpu().numpy().T
    frame = pd.DataFrame(Xfm.T, columns=[f"pixel_{i}" for i in range(F)], copy=False)

    dataset = Dataset(name="bench_dataset", targets=["target"])

    @dataset.reader
    def reader() -> pd.DataFrame:  # fixes the dataset's datatype (features arrive through Model.predict(features=...))
        return frame

    if kind == "mlp":
        module = torch_module(arrs)
        ModuleT = type(module)
        app = Model(name="bench_model", init=ModuleT, dataset=dataset)

        @app.predictor
        def predictor(m: ModuleT, features: pd.DataFrame) -> List[float]:
            return mlp_argmax(m, features)

        model_object = module
    else:
        from sklearn.linear_model import LogisticRegression

        est = sklearn_estimator(arrs, F)
        est.feature_names_in_ = np.asarray(frame.columns, dtype=object)
        app = Model(name="bench_model", init=LogisticRegression, dataset=dataset)

        @app.predictor
        def predictor(estimator: LogisticRegression, features: pd.DataFrame) -> List[float]:
            return linear_argmax(estimator, features)

        model_object = est
    from unionml_b200.model import ModelArtifact

    app.artifact = ModelArtifact(model_object)
    api_t, out = [], None
    for i in range(args.e2e_steps + 1):
        out = None  # the previous step's list is released outside the timed region (both arms do this)
        barrier()
        t0 = time.perf_counter()
        out = app.predict(features=frame)
        dt = time.perf_counter() - t0
        if i > 0:
            api_t.append(dt)
    got = np.asarray(out[: min(e2e_rows, 200_000)])
    classes = np.asarray(arrs.get("classes", np.arange(cfg["C"])), dtype=np.float64)
    want = classes[labels_all[lo : lo + got.shape[0]].cpu().numpy()]
    if not np.array_equal(got, want):
        raise SystemExit("bench: Model.predict(features=frame) labels differ from the resident path's")
    api_s = statistics.mean(api_t)
    from unionml_b200.predictors import last_call_stats

    api_stats = last_call_stats()

    # engine leg (round-1 e2e): pinned fp32 rows -> int32 labels in pinned memory
    eng_s, eng_stats = None, None
    if X_host is not None:
        labels_host = eng.pinned_empty(rows, np.int32)
        ts = []
        for i in range(args.e2e_steps + 1):
            barrier()
            t0 = time.perf_counter()
            if kind == "mlp":
                b = eng.stage(X_host, keep_f64=False)
                _, eng_stats = eng.predict_mlp(model, b, exact=True)
                b.free()
                eng_stats = dict(eng_stats, h2d_bytes=rows * F * 4, d2h_bytes=rows * 4)
            else:
                _, eng_stats = eng.predict_host(model, X_host, exact=True, out=labels_host)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if i > 0:
                ts.append(dt)
        eng_s = statistics.mean(ts)

    def max_over_ranks(v):
        if world > 1 and v is not None:
            t = torch.tensor([v], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    api_s, eng_s = max_over_ranks(api_s), max_over_ranks(eng_s)
    total = e2e_rows * world
    e2e = {
        "value": total / api_s, "unit": UNIT,
        # bytes that crossed PCIe, from the engine's own counters of the last call (the digits frame is integer-valued
        # float64: the gather threads narrow it to fp32 after checking every value; labels come back as int32)
        "h2d_bytes_per_step": int(api_stats.get("h2d_bytes", e2e_rows * F * 8)) * world,
        "d2h_bytes_per_step": int(api_stats.get("d2h_bytes", e2e_rows * 4)) * world,
        "source_bytes_per_step": int(e2e_rows * F * 8) * world,
        "ms_per_step": api_s * 1e3, "steps": args.e2e_steps, "rows_per_step": total,
        "path": "float64 feature-major pandas DataFrame (pageable) -> Model.predict(features=frame) -> @model.predictor "
                + ("mlp_argmax" if kind == "mlp" else "linear_argmax")
                + " -> host threads gather chunks into pinned bounce buffers (float64 -> fp32 when every value of the chunk "
                "survives it) -> H2D -> GPU transpose/down-cast -> scoring kernel (+fp64 re-score) -> D2H int32 labels -> "
                "List[float] filled from the class table while the batch is in flight",
        "sample": None if cfg["data"] == "digits" else f"{e2e_rows} rows of each rank's shard per step (the 50M x 784 batch does not fit in host memory)",
    }
    if eng_s is not None:
        e2e["engine_pinned_f32"] = {
            "value": rows * world / eng_s, "unit": UNIT, "ms_per_step": eng_s * 1e3,
            "h2d_bytes_per_step": int(eng_stats["h2d_bytes"]) * world, "d2h_bytes_per_step": int(eng_stats["d2h_bytes"]) * world,
            "path": "pinned fp32 C-order rows -> Engine.predict_host / stage+predict_mlp -> int32 labels in host memory (the round-1 e2e leg)",
        }
    return e2e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"],
                    help="N > 1: strong = ONE batch split across the GPUs (default), weak = the batch size per GPU")
    ap.add_argument("--rows", type=int, default=0, help="override: global rows (strong) / rows per GPU (weak)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-rows", type=int, default=0, help="bounded CPU sample (rows); default per config")
    ap.add_argument("--check-rows", type=int, default=200_000, help="rows per rank checked against float64 numpy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling only: skip the host-buffer legs")
    ap.add_argument("--gather", default="auto", choices=["auto", "fused", "push", "push4", "nccl"],
                    help="label exchange for --gpus > 1 (auto: short in-process A/B, fastest wins, all reported)")
    ap.add_argument("--no-multicast", action="store_true", help="per-peer stores instead of the NVLS multicast alias")
    ap.add_argument("--no-graph", action="store_true", help="N > 1: launch every step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--traffic", type=float, default=None, help="dram bytes/launch from a committed ncu capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the labels of the last timed step to DIR/labels.npy (float32; a seeded sample of large batches)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    args.scaling_resolved = "strong" if args.scaling in ("auto", "strong") else "weak"
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference_arm(args, cfg)
    return run_gpu_arm(args, cfg)


if __name__ == "__main__":
    sys.exit(main())
