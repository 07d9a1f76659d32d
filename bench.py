#!/usr/bin/env python
"""Benchmark of the KernelSHAP hot path: instances explained / second (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA engine (N > 1: run under torchrun)
  python bench.py --impl reference [...]                         the reference's CPU path on the host cores

Workload (config[1] of BASELINE.json): Adult-shaped synthetic tabular data (the real pickles need the network),
D = 49 encoded columns in 12 groups, 100 background rows, 2-class multinomial logistic regression, logit link,
nsamples = 2048, l1_reg = False; 2560 instances per GPU (weak scaling: every rank explains its own 2560).

A "step" explains the 2560 instances once.  ``value`` times steps with the inputs resident in HBM (CUDA events on
the engine's stream, L2 flushed between steps); ``e2e`` times the same step through the reference-facing plug-in
(`KernelShap._explainer.get_explanation`, i.e. the dks_explain_host C-ABI call) from pinned HOST buffers, including
the H2D copy of X and the D2H copy of the shap values.  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import statistics
import sys
import time

# One BLAS/OpenMP thread per process, set BEFORE NumPy is imported anywhere (this process and every spawned worker
# re-import this module, so they inherit it): a CPU worker stands for one single-CPU ray actor (distributed.py:125),
# and N workers with full-width BLAS pools would oversubscribe the host.  torchrun exports OMP_NUM_THREADS=1 itself;
# a plain `python bench.py` now behaves the same.
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
    os.environ[_v] = "1"

import numpy as np  # noqa: E402

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

N_INSTANCES = 2560
N_BACKGROUND = 100
NSAMPLES = 2048
METRIC = "instances explained/sec (bg=100, nsamples=2048) at 1/2/4/8 B200 vs ray CPU"
try:                                               # BASELINE.json's metric string, verbatim
    with open(os.path.join(REPO, "BASELINE.json")) as _f:
        METRIC = json.load(_f).get("metric", METRIC)
except (OSError, ValueError):
    pass


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "simt", "tcgen05", "shared"])
    ap.add_argument("--plan-mode", default="shared", choices=["shared", "per_instance"],
                    help="shared: one coalition plan per M for all instances (default, the headline); per_instance: a fresh "
                         "plan per instance drawn on the GPU (what shap does on the CPU)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the bounded CPU-oracle timing")
    ap.add_argument("--no-other-mode", action="store_true", help="skip the secondary leg (the other plan mode)")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the bounded runs of BASELINE configs[2]-[4]")
    ap.add_argument("--cpu-sample", type=int, default=16, help="instances the CPU baseline explains")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/shap_values.npy (float64, "
                         "[classes, instances of all ranks, groups]), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA engine (--impl ours)")
    return args


def workload(rank=0):
    """Adult-shaped problem; bg/model identical on every rank, the instances differ per rank (seed + rank)."""
    from distributedkernelshap_b200.datasets import adult_like
    base = adult_like(n_explain=N_INSTANCES, n_background=N_BACKGROUND, seed=0)
    if rank > 0:
        other = adult_like(n_explain=N_INSTANCES, n_background=N_BACKGROUND, seed=1000 + rank)
        base["X_explain"] = other["X_explain"]
    return base


def config_dict(world, kernel, plan_mode="shared", collective="none"):
    return {"workload": "Adult-shaped synthetic LR (BASELINE.json configs[1]): 2560 instances/GPU, D=49, 12 groups, "
                        "bg=100, nsamples=2048, l1_reg=False, logit link",
            "instances_per_gpu": N_INSTANCES, "global_instances": N_INSTANCES * world, "background": N_BACKGROUND,
            "nsamples": NSAMPLES, "features": 49, "groups": 12,
            "plan": PLAN_LABEL[plan_mode],
            "parallelism": f"dp{world} (instances sharded, one all-gather of phi)", "collective": collective, "kernel": kernel,
            "l2_flush_between_steps": True}


# ------------------------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_init():
    """Once per worker process: pin BLAS to one thread (belt and braces on top of the environment), build the workload
    and the explainer replica -- what a ray actor does in its constructor (kernel_shap.py:225-229), outside every timed
    region."""
    try:
        from threadpoolctl import threadpool_limits
        _CPU["limits"] = threadpool_limits(limits=1)
    except Exception:                                  # pragma: no cover - threadpoolctl is optional
        pass
    from oracle.shap_kernel_oracle import DenseData, KernelExplainerWrapperOracle
    wl = workload()
    dd = DenseData(wl["background"], wl["group_names"], wl["groups"])
    _CPU["X"] = wl["X_explain"]
    _CPU["explainer"] = KernelExplainerWrapperOracle(wl["predictor"].predict_proba, dd, link="logit", seed=0,
                                                     faithful_run=True)


def _cpu_worker(args):
    """Explain a slice of instances with the oracle in a single-threaded worker (one ray actor = one CPU); a fresh
    coalition plan per instance from the worker's own MT19937 stream, like the reference.  Returns the explain time."""
    if "explainer" not in _CPU:
        _cpu_init()
    lo, hi = args
    t0 = time.perf_counter()
    _CPU["explainer"].get_explanation(_CPU["X"][lo:hi], nsamples=NSAMPLES, l1_reg=False, silent=True)
    return time.perf_counter() - t0


def _blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([int(m.get("num_threads", 1)) for m in threadpool_info()] + [1])
    except Exception:                                  # pragma: no cover
        return None


def cpu_baseline_single(sample):
    """One worker, `sample` instances (== reference `--workers 1`; ~0.4 s per instance)."""
    t = _cpu_worker((0, sample))
    return {"value": sample / t, "unit": "instances/s", "cores": 1, "kind": "port", "blas_threads": _blas_threads(),
            "sample": f"first {sample} of the 2560 instances, oracle/shap_kernel_oracle.py (NumPy restatement of "
                      f"shap 0.35.0 KernelExplainer, interpreted S x N reduction loop kept, a fresh plan per instance), "
                      f"1 process, 1 BLAS thread, {t:.1f} s"}


def reference_config(cores, per_worker):
    return {"workload": "Adult-shaped synthetic LR (BASELINE.json configs[1]): D=49, 12 groups, bg=100, nsamples=2048, "
                        "l1_reg=False, logit link",
            "instances_per_step": cores * per_worker, "background": N_BACKGROUND, "nsamples": NSAMPLES, "features": 49,
            "groups": 12, "plan": "per instance (MT19937 stream of each worker, like shap)",
            "parallelism": f"{cores} single-threaded worker processes x {per_worker} instances (the ray ActorPool of "
                           "distributed.py:125 without ray)", "kernel": "cpu-oracle"}


def usable_cores():
    """Host cores this process may actually use: the CPU count, the scheduler affinity and the cgroup CPU quota, whichever is
    smallest (a container that shows 128 CPUs under a 24-CPU quota runs 128 busy workers SLOWER than 24: measured on this
    pool, scripts/cpu_scaling_probe.py)."""
    import math
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, math.ceil(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, math.ceil(quota / period)))
        except (OSError, ValueError):
            pass
    return n


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; shap/ray are not installable offline) on all host
    cores, one single-threaded worker process per core like the ray ActorPool (distributed.py:125).  Workers build
    their explainer replica once (pool initializer); a step is one pool.map over `cores` slices, wall-clock timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = usable_cores()
    per_worker = 4
    ctx = mp.get_context("spawn")
    times = []
    with ctx.Pool(cores, initializer=_cpu_init) as pool:
        pool.map(_cpu_worker, [(0, 1)] * cores)            # every worker is up and has imported/built everything
        for step in range(args.warmup + args.steps):
            chunks = [(w * per_worker, (w + 1) * per_worker) for w in range(cores)]
            t0 = time.perf_counter()
            pool.map(_cpu_worker, chunks, chunksize=1)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
    per_step = cores * per_worker
    ms = 1e3 * sum(times) / len(times)
    value = per_step / (ms / 1e3)
    sample = (f"{per_step} instances per step ({per_worker} per worker process x {cores} single-threaded workers, BLAS "
              f"pinned to 1 thread before NumPy loads) of the Adult-shaped workload; oracle port of shap 0.35.0 (faithful "
              "interpreted reduction loop, a fresh plan per instance)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "instances/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": reference_config(cores, per_worker),
            "cpu_baseline": {"value": value, "unit": "instances/s", "cores": cores, "kind": "port", "sample": sample,
                             "blas_threads": _blas_threads(), "cpu_count": os.cpu_count(),
                             "cores_note": "cores = min(cpu count, scheduler affinity, cgroup CPU quota)"},
            "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU in a background thread (NVML, every ~2 ms) while the timed
    region runs."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device, interval=0.002):
        self.device = device
        self.interval = interval
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = False
        self._thread = None

    def _run(self):
        import pynvml
        h = self._handle
        while not self._stop:
            try:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                bits = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.interval)

    def start(self):
        try:
            import threading
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[self.device]) if visible and visible.split(",")[0].isdigit() else self.device
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM)
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self._thread is None:
            return out
        self._stop = True
        self._thread.join(timeout=2)
        if self.samples:
            out.update(sm_mhz=statistics.median(self.samples), reasons=sorted(self.reasons), samples=len(self.samples))
        return out


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
def measure_mode(wl, X, plan_mode, kernel, steps, warmup, flush, stream):
    """Device-resident and end-to-end throughput of one plan mode on one GPU (the secondary leg of the default line):
    same step, same timing rules (CUDA events on the engine's stream, L2 flushed between steps)."""
    import torch
    from distributedkernelshap_b200.explainers.kernel_shap import KernelShap
    n, D = X.shape
    explainer = KernelShap(wl["predictor"].predict_proba, link="logit", feature_names=wl["group_names"], seed=0,
                           plan_mode=plan_mode)
    explainer.fit(wl["data"]["background"]["X"]["preprocessed"], group_names=wl["group_names"], groups=wl["groups"])
    engine = explainer._explainer
    engine.set_kernel(kernel)
    G, C = engine.data.groups_size, engine.D
    engine.get_explanation(X, nsamples=NSAMPLES, l1_reg=False, silent=True)       # plans built + uploaded
    engine.set_stream(stream.cuda_stream)
    X_dev = torch.from_numpy(X).cuda()
    phi_dev = torch.empty((C, n, G), dtype=torch.float64, device="cuda")
    for _ in range(warmup):
        flush.zero_()
        engine.explain_device(X_dev.data_ptr(), n, phi_dev.data_ptr(), nsamples=NSAMPLES)
    engine.check_status()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    torch.cuda.synchronize()
    for k in range(steps):
        flush.zero_()
        starts[k].record(stream)
        engine.explain_device(X_dev.data_ptr(), n, phi_dev.data_ptr(), nsamples=NSAMPLES)
        ends[k].record(stream)
    torch.cuda.synchronize()
    engine.check_status()
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps
    X_pin = torch.empty((n, D), dtype=torch.float64).pin_memory()
    X_pin.copy_(torch.from_numpy(X))
    X_host = X_pin.numpy()
    for _ in range(2):
        engine.get_explanation(X_host, nsamples=NSAMPLES, l1_reg=False, silent=True)
    torch.cuda.synchronize()
    blocks = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            engine.get_explanation(X_host, nsamples=NSAMPLES, l1_reg=False, silent=True)
        torch.cuda.synchronize()
        blocks.append(time.perf_counter() - t0)
    e2e = n * steps / statistics.median(blocks)
    out = {"plan": PLAN_LABEL[plan_mode], "value": n / (ms / 1e3), "unit": "instances/s", "ms_per_step": ms,
           "e2e": {"value": e2e, "unit": "instances/s", "h2d_bytes_per_step": n * D * 8, "d2h_bytes_per_step": C * n * G * 8},
           "kernel_ms": engine.last_timings_ms()["coalitions"]}       # the host-path call above: plain launches
    engine.close()
    return out


OTHER_CONFIGS = {
    "configs[2]": dict(label="synthetic dense tabular: 64 features (ungrouped), bg=512, nsamples=4096, LR (BASELINE.json "
                             "configs[2]; 16384 of its 1M instances)", kind="dense", features=64, bg=512, ns=4096),
    "configs[3] grouped": dict(label="wide one-hot, grouped reading: 64 variables x 16 levels = 1024 columns, bg=256, "
                                     "nsamples=8192 (BASELINE.json configs[3]; 8192 of its 100k instances)", kind="onehot",
                               features=1024, bg=256, ns=8192),
    "configs[3] singleton": dict(label="wide one-hot, singleton reading: each of the 1024 one-hot columns its own group "
                                       "(M = 1024: sixteen-word coalition rows, projection solve with a 1023 x 1023 normal "
                                       "matrix factored once per plan on the host), uniform level probabilities, bg=256, "
                                       "nsamples=8192 (BASELINE.json configs[3]; 2048 of its 100k instances); l1_reg=False "
                                       "(feature selection is refused above 128 groups)", kind="onehot_singleton",
                                 features=1024, bg=256, ns=8192, l1=False),
    "configs[4] one GPU": dict(label="synthetic: 128 features (two-word coalition rows), bg=512, nsamples=4096 (BASELINE.json "
                                     "configs[4]; 16384 instances = a slice of one GPU's share of the 10M)", kind="dense",
                               features=128, bg=512, ns=4096),
}


def measure_config(name, spec, flush, stream, steps=3, warmup=2):
    """Throughput of one of the other BASELINE.json configs at a bounded instance count on one GPU (shared plans): device
    resident (CUDA events, L2 flushed between steps), through the host API with l1_reg=False, and through the host API with
    the reference's DEFAULT kwargs (l1_reg='auto': LassoLarsIC feature selection on the device, csrc/dks_l1.cuh)."""
    import torch
    from distributedkernelshap_b200.data import DenseData
    from distributedkernelshap_b200.datasets import dense_tabular, wide_onehot
    from distributedkernelshap_b200.engine import GpuKernelExplainer
    n = {"dense": 16384, "onehot": 8192, "onehot_singleton": 2048}[spec["kind"]]
    wl = dense_tabular(n, spec["features"], spec["bg"], seed=0) if spec["kind"] == "dense" else \
        wide_onehot(n, 64, 16, spec["bg"], seed=0, singleton_groups=spec["kind"] == "onehot_singleton")
    X = np.ascontiguousarray(wl["X_explain"])
    eng = GpuKernelExplainer(wl["predictor"].predict_proba, DenseData(wl["background"], wl["group_names"], wl["groups"]),
                             link="logit", seed=0)
    G = len(wl["groups"])
    eng.shap_values(X[:512], nsamples=spec["ns"], l1_reg=False)              # plans built + uploaded
    eng.set_stream(stream.cuda_stream)
    X_dev = torch.from_numpy(X).cuda()
    phi = torch.empty((2, n, G), dtype=torch.float64, device="cuda")
    ms = []
    for k in range(warmup + steps):       # two warm-up steps: the first runs plainly, the second captures the CUDA graph
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.explain_device(X_dev.data_ptr(), n, phi.data_ptr(), nsamples=spec["ns"])
        e1.record(stream)
        torch.cuda.synchronize()
        if k >= warmup:
            ms.append(e0.elapsed_time(e1))
    eng.check_status()
    out = {"workload": spec["label"], "instances": n, "plan": "shared per M", "value": n / (statistics.mean(ms) / 1e3),
           "unit": "instances/s", "ms_per_step": statistics.mean(ms)}
    eng.shap_values(X, nsamples=spec["ns"], l1_reg=False)                    # untimed: staging buffers of this size allocated
    dts = []
    for _ in range(3):
        t0 = time.perf_counter()
        eng.shap_values(X, nsamples=spec["ns"], l1_reg=False)
        dts.append(time.perf_counter() - t0)
    out["e2e"] = {"value": n / statistics.median(dts), "unit": "instances/s", "l1_reg": False,
                  "timing": "host API, host arrays in and out; median of three calls after one warm-up call"}
    if not spec.get("l1", True):
        eng.close()
        return out
    n1 = 2048
    try:
        eng.shap_values(X[:64], nsamples=spec["ns"])                          # l1 tables uploaded
        dts = []
        for _ in range(3):
            t0 = time.perf_counter()
            sv = eng.shap_values(X[:n1], nsamples=spec["ns"])                 # reference default: l1_reg='auto'
            dts.append(time.perf_counter() - t0)
        out["e2e_reference_default_kwargs"] = {
            "value": n1 / statistics.median(dts), "unit": "instances/s", "instances": n1, "l1_reg": "auto (LassoLarsIC aic)",
            "timing": "median of three host-API calls",
            "mean_features_selected": float(np.count_nonzero(sv[1], axis=1).mean())}
    except Exception as exc:                                                  # pragma: no cover - reported, not hidden
        out["e2e_reference_default_kwargs"] = {"error": repr(exc)[:300]}
    eng.close()
    return out


PLAN_LABEL = {"shared": "shared per M (one plan for every instance with M varying groups; the engine's fast mode)",
              "per_instance": "per instance, drawn on the GPU (Philox keyed by seed and global row: what shap does on the CPU)"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from distributedkernelshap_b200 import parallel
    from distributedkernelshap_b200.explainers.kernel_shap import KernelShap

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one process per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    wl = workload(rank)
    X = np.ascontiguousarray(wl["X_explain"], dtype=np.float64)
    n, D = X.shape
    # the reference's call sequence (benchmarks/ray_pool.py:34-37); under torchrun distributed_opts selects the SPMD path
    dopts = {"n_cpus": world, "batch_size": None, "actor_cpu_fraction": 1.0} if world > 1 else None
    explainer = KernelShap(wl["predictor"].predict_proba, link="logit", feature_names=wl["group_names"], seed=0,
                           distributed_opts=dopts, plan_mode=args.plan_mode)
    explainer.fit(wl["data"]["background"]["X"]["preprocessed"], group_names=wl["group_names"], groups=wl["groups"])
    plugin = explainer._explainer                       # DistributedExplainer (N > 1) or the engine itself
    engine = plugin.pool[0] if world > 1 else plugin
    engine.set_kernel(args.kernel)
    G, C = engine.data.groups_size, engine.D

    # first call builds + uploads the shared plans (one per M present) -- outside every timed region
    sv0 = engine.get_explanation(X, nsamples=NSAMPLES, l1_reg=False, silent=True)

    # ---------------- device-resident steps: `value` ----------------
    stream = torch.cuda.Stream()                 # not the legacy default stream: the engine replays its launch sequence
    torch.cuda.set_stream(stream)                # as one CUDA graph only on a capturable stream
    engine.set_stream(stream.cuda_stream)
    X_dev = torch.from_numpy(X).cuda()
    phi_dev = torch.empty((C, n, G), dtype=torch.float64, device="cuda")
    phi_all = torch.empty((world, C, n, G), dtype=torch.float64, device="cuda") if world > 1 else None
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB of L2
    # N > 1: the all-gather of phi is the engine's own push over NVLink peer memory (each rank stores its block into every
    # peer's gathered buffer, then one cross-GPU barrier); NCCL all_gather_into_tensor if peer memory cannot be mapped
    gather, collective = None, "none"
    if world > 1:
        collective = "nccl all_gather_into_tensor"
        # after the solve the engine's push kernel stores this rank's phi block into all peers' gathered buffers over NVLink peer
        # memory (128-bit coalesced stores) and the explain call ends with the engine's own flag exchange (signal + wait per
        # peer).  Measured on an 8-GPU box (profiles/r2_bench_8gpu_d_*): 0.185 ms/step at N=8 against 0.200 with
        # ncclAllGather and 0.210 with the stores issued from the fused kernel's epilogue (DKS_PUSH_IN_KERNEL=1).
        # DKS_BENCH_NCCL=1 forces NCCL, DKS_BENCH_SYMM_BARRIER=1 the symmetric-memory barrier instead of the flags.
        use_push = os.environ.get("DKS_BENCH_NCCL", "0") != "1"
        if use_push:
            try:
                own_sync = os.environ.get("DKS_BENCH_SYMM_BARRIER", "0") != "1"
                gather = parallel.PeerGather(engine, C, n, G, torch.device("cuda", local_rank), own_sync=own_sync)
                phi_dev = gather.local
                how = "the fused kernel's epilogue" if os.environ.get("DKS_PUSH_IN_KERNEL", "0") == "1" else "the engine's push kernel"
                collective = (f"phi stored into every peer's gathered buffer by {how} (NVLink peer memory) + " +
                              ("the engine's flag exchange" if own_sync else "symmetric-memory barrier"))
            except Exception as exc:                      # pragma: no cover - depends on the box
                print(f"[bench] peer-memory gather unavailable ({exc!r}); using NCCL", file=sys.stderr)
                gather = None
        flags = torch.tensor([1 if gather is not None else 0], device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)      # all ranks or none
        if int(flags.item()) == 0 and gather is not None:
            gather.close()
            gather, phi_dev, collective = None, torch.empty((C, n, G), dtype=torch.float64, device="cuda"), \
                "nccl all_gather_into_tensor"

    def step_device():
        engine.explain_device(X_dev.data_ptr(), n, phi_dev.data_ptr(), nsamples=NSAMPLES)
        if gather is not None:
            gather.barrier()
        elif world > 1:
            dist.all_gather_into_tensor(phi_all, phi_dev)

    if gather is not None:                                # once: the pushed result equals NCCL's
        step_device()
        torch.cuda.synchronize()
        dist.all_gather_into_tensor(phi_all, phi_dev.contiguous())
        torch.cuda.synchronize()
        assert torch.equal(gather.buffer, phi_all), "peer-memory gather differs from all_gather_into_tensor"

    for _ in range(args.warmup):
        flush.zero_()
        step_device()
    engine.check_status()
    launches0 = engine.kernel_launches()
    kernel_ms = []
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank, interval=0.002 if world == 1 else 0.02)   # N ranks share the host's CPU quota
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    # The K steps are enqueued behind a short device-side sleep, so the GPU executes them back to back from a full queue: a
    # host hiccup while enqueueing (N ranks share the box's CPU quota; measured: single steps of 2-8 ms on an otherwise
    # 0.2 ms step, on a box whose load average was 14-20 before the job started) would otherwise idle the GPU inside the
    # device-timed region.  Every step is still timed with its own pair of CUDA events; the sleep ends before the first
    # start event.
    torch.cuda._sleep(int((0.004 if world == 1 else 0.020) * 1.9e9))
    if world > 1:
        # ... and the ranks' GPUs are aligned by one tiny collective on the stream AFTER the sleep, so a rank whose host was
        # late to start enqueueing does not show up as a long first step on its peers
        dist.all_reduce(torch.zeros(1, device="cuda"))
    for k in range(args.steps):
        flush.zero_()
        starts[k].record(stream)
        step_device()
        ends[k].record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    engine.check_status()
    launches = engine.kernel_launches() - launches0
    # what the last timed step handed its caller: this rank's phi block, or the gathered phi of every rank (N > 1)
    if args.dump_outputs and rank == 0:
        last_phi = (phi_dev if world == 1 else gather.buffer if gather is not None else phi_all).cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "shap_values.npy"),
                last_phi.reshape(world, C, n, G).transpose(1, 0, 2, 3).reshape(C, world * n, G))
    # per-kernel device time (CUDA events around the coalition stage): three extra steps with plain launches -- the replayed
    # graph of the timed region carries no timing nodes
    engine.set_option("graph", 0)
    for _ in range(3):
        flush.zero_()
        step_device()
        kernel_ms.append(engine.last_timings_ms()["coalitions"])
    engine.set_option("graph", 1)
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / args.steps
    value = world * n / (ms_per_step / 1e3)
    step_spread = {"min": min(step_ms), "median": statistics.median(step_ms), "max": max(step_ms)}     # this rank's steps
    np.testing.assert_allclose(phi_dev[1].cpu().numpy(), sv0[1], rtol=0, atol=1e-12)   # same values as the host path

    if gather is not None:
        gather.close()                      # the host-API path below gathers with NCCL on device-resident blocks (no peer stores)
        gather = None
    # ---------------- end to end through the plug-in with host buffers: `e2e` ----------------
    X_pin = torch.empty((world * n if world > 1 else n, D), dtype=torch.float64).pin_memory()
    if world > 1:
        gathered = [torch.empty((n, D), dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(gathered, X_dev)
        X_pin.copy_(torch.cat(gathered).cpu())
    else:
        X_pin.copy_(torch.from_numpy(X))
    X_host = X_pin.numpy()
    for _ in range(max(2, args.warmup // 2)):
        plugin.get_explanation(X_host, nsamples=NSAMPLES, l1_reg=False, silent=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    # K steps per block, wall clock; the blocks are milliseconds long, so the median of five blocks is reported (one block is
    # at the mercy of a host hiccup)
    blocks = []
    for _ in range(5):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = plugin.get_explanation(X_host, nsamples=NSAMPLES, l1_reg=False, silent=True)
        torch.cuda.synchronize()
        blocks.append(time.perf_counter() - t0)
    e2e_s = torch.tensor([statistics.median(blocks)], dtype=torch.float64, device="cuda")
    # what came back through the host API is what the device-resident path computed (this rank's rows of the gathered result)
    np.testing.assert_allclose(np.asarray(out[1])[rank * n:(rank + 1) * n], sv0[1], rtol=0, atol=1e-12)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.steps / float(e2e_s.item())
    h2d = n * D * 8
    d2h = C * n * G * 8

    # ---------------- sustained: back-to-back steps for ~2 s (a clock record with more than one sample) ----------------
    sustained = None
    if world == 1:
        reps = max(200, int(2000.0 / max(ms_per_step, 1e-3)))
        sam2 = ClockSampler(local_rank)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        sam2.start()
        ev0.record(stream)
        for _ in range(reps):
            step_device()
        ev1.record(stream)
        torch.cuda.synchronize()
        ck = sam2.stop()
        engine.check_status()
        sus_ms = ev0.elapsed_time(ev1) / reps
        sustained = {"steps": reps, "seconds": ev0.elapsed_time(ev1) / 1e3, "ms_per_step": sus_ms, "value": n / (sus_ms / 1e3),
                     "l2": "warm (no flush between steps)",
                     "clocks": {"sm_mhz": ck["sm_mhz"], "sm_max_mhz": ck["sm_max_mhz"], "reasons": ck["reasons"],
                                "samples": ck["samples"]}}

    # ---------------- the other plan mode (same timing rules), so that the driver's record holds both ----------------
    other = None
    if world == 1 and not args.no_other_mode:
        other_mode = "per_instance" if args.plan_mode == "shared" else "shared"
        other = measure_mode(wl, X, other_mode, args.kernel, args.steps, args.warmup, flush, stream)

    # ---------------- the other BASELINE.json configs at a bounded size (coverage data points in the same record) --------
    other_configs = None
    if world == 1 and not args.no_other_configs:
        other_configs = {}
        for cname, spec in OTHER_CONFIGS.items():
            try:
                other_configs[cname] = measure_config(cname, spec, flush, stream)
            except Exception as exc:                                          # pragma: no cover
                other_configs[cname] = {"error": repr(exc)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (fused coalition kernel) ----------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    alg_bytes = 4.0 * NSAMPLES * N_BACKGROUND * D * n            # SURVEY §8(d): B_alg = 4*S*N*D per instance
    k_ms = statistics.mean(kernel_ms) if kernel_ms else ms_per_step
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(REPO, "profiles", "roofline_traffic.json"))).get("dram_bytes_per_launch")
    except Exception:
        pass
    elems = float(NSAMPLES) * N_BACKGROUND * n                   # sigmoid evaluations per launch (T_alg)
    sm_mhz = clocks.get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    mufu_peak = 148 * 16 * sm_mhz * 1e6                          # MUFU ops/s at the observed clock (16 lanes/clk/SM, measured)
    fused_names = "explain_shared_fused_kernel (shared-plan path: coalition sums + link + projection solve in one kernel; tcgen05 kernel on a side stream for partial varying sets)"
    kname, mufu_per_elem = {
        "auto": (fused_names, 0.5), "shared": (fused_names, 0.5),
        "tcgen05": ("explain_tcgen05_kernel", 1.5), "simt": ("explain_simt_kernel", 2.0)}[engine.kernel]
    if args.plan_mode == "per_instance" and engine.kernel != "simt":
        kname, mufu_per_elem = "sample_plans_kernel + factor_plans_kernel + explain_tcgen05_kernel (per-instance plans)", 1.5
    mufu_ops = mufu_per_elem * elems / (k_ms * 1e-3)
    # The pipe that binds this stage is the MUFU (XU) pipe -- neither HBM nor the tensor pipe: `frac` is measured against
    # it.  The effective-HBM figure SURVEY §8(d) defines (bytes of the reference-shaped masked batch / kernel time) is kept
    # as a secondary field: the fused kernels never materialise that batch, so it exceeds the HBM peak by design.
    roofline = {"bound": "mufu", "achieved": mufu_ops / 1e9, "peak": mufu_peak / 1e9, "unit": "Gop/s (MUFU lane-ops)",
                "frac": mufu_ops / mufu_peak, "traffic": traffic, "kernel": kname, "kernel_ms": k_ms,
                "peak_source": "148 SMs x 16 MUFU lanes/clk (measured, profiles/r1_mufu_probe_b200.txt) x the SM clock sampled "
                               "during the timed region",
                "mufu_ops_per_elem": mufu_per_elem, "elems_per_launch": elems,
                "effective_hbm": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                  "peak_source": peak_src,
                                  "note": "algorithmic bytes of the masked batch (4*S*N*D per instance, SURVEY §8d) / kernel "
                                          "time; an EFFECTIVE figure (> 1 expected): the batch is never materialised"},
                "traffic_note": "dram__bytes_read + dram__bytes_write of the dominant kernel per launch, ncu --set full "
                                "(profiles/roofline_traffic.json)"}
    if engine.kernel in ("auto", "shared") and args.plan_mode == "shared":
        # 7 packed fp32 ops (FFMA2/FMUL2/FADD2: two lanes each, two issue cycles) per four sigmoids = 3.5 fp32 lane-ops per
        # element against 128 lanes/clk/SM
        fp32_peak = 148 * 128 * sm_mhz * 1e6
        roofline.update({"fp32_lane_ops_per_elem": 3.5, "fp32_pipe_frac": 3.5 * elems / (k_ms * 1e-3) / fp32_peak})

    line = {"metric": METRIC, "value": value, "unit": "instances/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 sigmoid/accumulate, f64 link + WLS", "data": "synthetic",
            "config": config_dict(world, engine.kernel, args.plan_mode, collective),
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"],
                       "samples": clocks["samples"]},
            "e2e": {"value": e2e_value, "unit": "instances/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "KernelShap._explainer.get_explanation -> dks_explain_host (pinned host X in, host phi out); N > 1: "
                           "DistributedExplainer under torchrun (phi stays on the device through the all-gather, one D2H)",
                    "timing": f"median of 5 blocks of {args.steps} calls, wall clock, max over ranks"},
            "gpu_launches": int(launches), "step_ms_rank0": step_spread, "roofline": roofline}
    if sustained is not None:
        line["sustained"] = sustained
    if other is not None:
        line["per_instance" if args.plan_mode == "shared" else "shared_plan"] = other
    if other_configs is not None:
        line["other_configs"] = other_configs
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_single(args.cpu_sample)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
