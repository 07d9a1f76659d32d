"""Throughput of the one-hidden-layer ReLU network path on one GPU: Adult-shaped data (2560 instances, 12 groups, bg = 100,
nsamples = 2048) explained through a seeded scikit-learn MLPClassifier of 100 ReLU units with a logistic output.

Device-resident steps (explain_device, CUDA events on the engine's stream, L2 overwritten between steps) for
  'auto'          shared plans, shared-plan MLP kernel (mlp_atab_kernel + mlp_shared_kernel) + projection solve;
  'simt'          shared plans, general MLP kernel for every instance;
  'per_instance'  a plan drawn on the device per instance, general MLP kernel.
Kernel times from torch.profiler in a separate run; the derived fp32 floor of the shared-plan kernel; parity of 8
instances against the CPU oracle given the same plans; the oracle's time per instance on one core.  Prints one JSON line
and, with ``--out``, writes it to that file as well.

    python scripts/gpu_mlp_bench.py [--steps 20] [--warmup 3] [--out FILE]
"""
import os

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):     # the oracle baseline runs on one core
    os.environ.setdefault(_v, "1")

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import time  # noqa: E402
import warnings  # noqa: E402

import numpy as np  # noqa: E402

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

NSAMPLES = 2048
H = 100
SMS, LANES = 148, 128                 # B200: SMs, fp32 lanes per SM and clock


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [f.strip() for f in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def workload():
    from sklearn.exceptions import ConvergenceWarning
    from sklearn.neural_network import MLPClassifier
    from distributedkernelshap_b200.datasets import adult_like
    d = adult_like()
    rng = np.random.default_rng(0)
    Xt = np.concatenate([d["background"], d["X_explain"]])
    y = (Xt[:, :4] @ rng.standard_normal(4) + Xt[:, 4:] @ rng.normal(0, 0.5, Xt.shape[1] - 4) > 0).astype(int)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)
        mlp = MLPClassifier(hidden_layer_sizes=(H,), max_iter=30, random_state=0).fit(Xt, y)
    return d, mlp


def engine(d, mlp, kernel, plan_mode):
    from distributedkernelshap_b200.data import DenseData
    from distributedkernelshap_b200.engine import GpuKernelExplainer
    return GpuKernelExplainer(mlp.predict_proba, DenseData(d["background"], d["group_names"], d["groups"]), link="logit",
                              seed=0, kernel=kernel, plan_mode=plan_mode)


def timed_steps(eng, X, steps, warmup, flush, stream):
    import torch
    n = X.shape[0]
    eng.shap_values(X, nsamples=NSAMPLES, l1_reg=False)            # plans built and uploaded
    eng.set_stream(stream.cuda_stream)
    X_dev = torch.from_numpy(X).cuda()
    phi = torch.empty((eng.D, n, eng.data.groups_size), dtype=torch.float64, device="cuda")
    for _ in range(warmup):                                        # plain run, graph capture, replays
        flush.zero_()
        eng.explain_device(X_dev.data_ptr(), n, phi.data_ptr(), nsamples=NSAMPLES)
    eng.check_status()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    torch.cuda.synchronize()
    for k in range(steps):
        flush.zero_()
        starts[k].record(stream)
        eng.explain_device(X_dev.data_ptr(), n, phi.data_ptr(), nsamples=NSAMPLES)
        ends[k].record(stream)
    torch.cuda.synchronize()
    eng.check_status()
    ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    med = statistics.median(ms)
    return {"instances_per_s": n / (med / 1e3), "ms_per_step_median": med, "ms_per_step_min": min(ms),
            "ms_per_step_max": max(ms), "steps": steps, "graph_launches": eng.graph_launches()}, phi


def kernel_times(eng, X, flush, steps=5):
    """Mean device time per step of every kernel, from torch.profiler (a run of its own, plain launches)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    eng.set_option("graph", 0)
    for _ in range(2):
        eng.shap_values(X, nsamples=NSAMPLES, l1_reg=False)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            flush.zero_()
            eng.shap_values(X, nsamples=NSAMPLES, l1_reg=False)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t <= 0:
            continue
        name = e.key.split("(")[0].split("<")[0].replace("void ", "").split("::")[-1]
        if "mlp" in e.key or "wls" in e.key or "sample" in e.key or "factor" in e.key:
            out[name] = out.get(name, 0.0) + t / 1e3 / steps        # ms per step
    eng.set_option("graph", 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    result = {"card": card(), "workload": "adult_like(): 2560 instances, 12 groups (49 columns), bg=100, nsamples=2048, "
                                          f"MLPClassifier(hidden_layer_sizes=({H},), relu, logistic output, random_state=0)",
              "l2": "256 MB buffer overwritten between timed steps"}
    d, mlp = workload()
    X = np.ascontiguousarray(d["X_explain"])
    n, N = X.shape[0], d["background"].shape[0]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.Stream()
    legs, phis = {}, {}
    for label, kernel, mode in (("auto", "auto", "shared"), ("simt", "simt", "shared"), ("per_instance", "auto", "per_instance")):
        eng = engine(d, mlp, kernel, mode)
        legs[label], phis[label] = timed_steps(eng, X, args.steps, args.warmup, flush, stream)
        if label == "auto":
            result["kernel_ms_auto"] = kernel_times(eng, X, flush)
            auto_eng = eng
        elif label == "simt":
            result["kernel_ms_simt"] = kernel_times(eng, X, flush)
            eng.close()
        else:
            eng.close()
    result["legs"] = legs
    a, s = phis["auto"].cpu().numpy(), phis["simt"].cpu().numpy()
    result["auto_vs_simt_max_rel"] = float((np.abs(a - s).max(axis=-1) / np.abs(s).max(axis=-1)).max())

    # derived fp32 floor of the shared-plan kernel: (unit, masked row) pairs x lane-ops per pair
    w2 = mlp.coefs_[1][:, 0]
    npos, nneg = int((w2 > 0).sum()), int((w2 < 0).sum())
    hp = ((npos + 7) // 8 * 8 + (nneg + 7) // 8 * 8 + 15) // 16 * 16
    S = min(NSAMPLES, 2 ** 12 - 2)
    pairs = n * S * N * H
    k = 2                                          # FADD a'+d', and per two units one FADD |x|+|y| plus the chunk's tree
    clock_ghz = float(result["card"]["max_sm_clock"].split()[0]) / 1e3
    floor_ms = pairs * k * hp / H / (SMS * LANES * clock_ghz * 1e9) * 1e3
    floor_ideal_ms = pairs * k / (SMS * LANES * clock_ghz * 1e9) * 1e3
    km = result["kernel_ms_auto"]
    coal_ms = km.get("mlp_shared_kernel", 0.0) + km.get("mlp_atab_kernel", 0.0)
    result["floor"] = {"pairs_per_step": pairs, "lane_ops_per_pair": k, "padded_units": hp, "hidden_units": H,
                       "clock_ghz": clock_ghz, "fp32_floor_ms_at_H": floor_ideal_ms, "fp32_floor_ms_as_built": floor_ms,
                       "coalition_kernels_ms": coal_ms,
                       "fraction_of_floor_at_H": floor_ideal_ms / coal_ms if coal_ms else None,
                       "fraction_of_floor_as_built": floor_ms / coal_ms if coal_ms else None}

    # parity against the oracle given the same plans, and the oracle's time per instance on one core
    from oracle.shap_kernel_oracle import DenseData, KernelExplainerOracle
    orc = KernelExplainerOracle(mlp.predict_proba, DenseData(d["background"], d["group_names"], d["groups"]), link="logit")
    M, _ = auto_eng.varying(X)
    worst, secs = 0.0, []
    for i in range(0, n, n // 8)[:8]:
        plan = auto_eng.shared_plan(int(M[i]), NSAMPLES)
        t0 = time.perf_counter()
        want = orc.explain(X[i:i + 1], plan=(plan.dense(), plan.weights), nsamples=NSAMPLES, l1_reg=False)
        secs.append(time.perf_counter() - t0)
        worst = max(worst, float(np.abs(a[1, i] - want[:, 1]).max() / np.abs(want[:, 1]).max()))
    result["parity_8_instances_max_rel"] = worst
    result["oracle_s_per_instance_one_core"] = statistics.median(secs)
    result["speedup_auto_vs_oracle_one_core"] = legs["auto"]["instances_per_s"] * statistics.median(secs)
    auto_eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
