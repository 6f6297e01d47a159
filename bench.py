#!/usr/bin/env python
"""Headline benchmark: fp64 GPR loss+grad evaluations per second at N=32768, D=8 on B200 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--num-points 32768] [--dump-outputs DIR]

One "step" = one full evaluation of model.loss() + loss.backward() for GPR with an Rbf-ARD kernel on the
synthetic regression problem of BASELINE.md section 3 (covariance build, Cholesky, solves, log-det, and the
analytic gradient through (L L^T)^-1).  Prints ONE JSON line (rank 0).

* value      : evaluations/s with X, Y resident in HBM, CUDA-event timed, max over ranks.  The loss of the timed
               steps is checked against the unmodified reference's value at this size
               (tests/golden/gpr_n32768_reference.json); the bench FAILS if it is off by more than 1e-9.
* e2e        : the same through the public API with HOST inputs, over all K steps: per step X, Y are copied from
               pinned host memory into the model, loss()+backward() run, loss and gradients are read back to the host.
* roofline   : the O(N^3) part (gpb potrf + potri, > 95 % DMMA GEMM kernel) against the FP64 tensor-pipe issue
               ceiling measured live (gpb_dmma_issue_probe); the live cuBLAS DGEMM figure is reported beside it
               (MEASURED_PEAKS.json carries no FP64 entry).
* cpu_baseline / --impl reference : the UNMODIFIED reference (baseline/_ref, pip-installed from /root/reference)
               on the host cores, all threads, on a bounded sample (the largest N of 4096..16384 whose steps fit the
               time budget); `value` extrapolates to the named N with the exponent measured on this pool between
               N=12288 and the full N=32768 run (tests/golden/gpr_n32768_reference.json: 124.9 s on 16 threads).
* vendor_baseline : the unmodified reference under model.cuda() on the same B200 (torch -> cuSOLVER/cuBLAS), the
               vendor-library bar of SURVEY 2.1, at the named size, CUDA-synchronised wall clock.
* sharded    : the configurations that shard (bench_sharded.py): VFE N=1e7 strong-scaled, SVGP data-parallel,
               distributed exact GPR -- with their collectives; at --gpus 1 the single-GPU figures of the same runs.
* --gpus N>1 : the headline GPR evaluation does not shard at this size (SURVEY 8e, DESIGN.md "replicas only"): every
               rank runs an independent replica; value = N * K / max-rank time.
* --steps K  : the number of timed steps of every block of the line: value, e2e, int8_sliced_experimental and each
               sharded configuration.
* --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned to its caller -- the loss
               and the gradient of every hyper-parameter -- as DIR/<name>.npy (float64), so that two builds can be
               compared output for output (the inputs are seeded: the same arguments give the same inputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fp64 GPR loss+grad evals/sec @N=32768,D=8; Cholesky FP64 TFLOP/s vs peak"
D_IN = 8
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
PIN_FILE = os.path.join(ROOT, "tests", "golden", "gpr_n32768_reference.json")
# host-CPU cost of the reference between the sample size and the named size, measured on this pool's box (16 threads):
# 7.79 s at N=12288 (BENCH_r01.json), 124.9 s at N=32768 (tests/golden/gpr_n32768_reference.json) -> exponent 2.83
CPU_SCALING_EXPONENT = float(np.log(124.891459346 / 7.785708919) / np.log(32768.0 / 12288.0))
# full-size seconds / sample seconds measured on this pool's box with the unmodified reference (16 threads): N=12288 7.79 and
# 8.42 s (BENCH_r01.json, profiles/r02_bench_first.json), N=16384 18.57 s (profiles/r02_bench_reference_arm_first.json),
# N=32768 124.89 s; sample sizes without a measured ratio fall back to the exponent
CPU_FULL_OVER_SAMPLE = {12288: 124.891459346 / 8.10, 16384: 124.891459346 / 18.57}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--num-points", dest="n", type=int, default=32768, help="training points (the named config is 32768)")
    ap.add_argument("--cpu-sample-n", type=int, default=0, help="reference sample size (0 = choose by time budget)")
    ap.add_argument("--cpu-budget-s", type=float, default=240.0, help="time budget of the --impl reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vendor-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--no-int8-sliced", action="store_true", help="skip the experimental int8-sliced engine block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and gradients of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def workload_config(n, world):
    """`config` of the JSON line -- identical for both arms (the reference arm samples THIS workload)."""
    return {"workload": "GPR Rbf-ARD fp64 N=%d D=%d dy=1 loss+grad (configs[1])" % (n, D_IN),
            "parallelism": "replicas only (x%d)" % world if world > 1 else "single GPU",
            "l2": "inputs_exceed_l2 (the N^2 covariance/factor buffer is %.1f GB)" % (8.0 * n * n / 1e9)}


def synth_regression(n, d, seed=1234):
    """SURVEY 8d's synthetic inputs (CPU generator, so the reference's loss pins apply): X ~ U[0,1)^d,
    Y = sin(X w) + 0.1 eps.  Stated here rather than imported: oracle/ is only the checker."""
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(n, d, generator=g, dtype=torch.float64)
    w = torch.randn(d, 1, generator=g, dtype=torch.float64)
    Y = torch.sin(X @ w) + 0.1 * torch.randn(n, 1, generator=g, dtype=torch.float64)
    return X, Y, g


def reference_pin(n):
    if n != 32768 or not os.path.exists(PIN_FILE):
        return None
    with open(PIN_FILE) as f:
        return json.load(f)


# ------------------------------------------------------------------------------------------------------
# The unmodified reference (baseline/_ref): host-CPU arm and vendor-library (model.cuda()) arm
# ------------------------------------------------------------------------------------------------------
def _reference_modules():
    """Import cics-nd/gptorch from baseline/_ref (never from this repo's package)."""
    import warnings
    warnings.filterwarnings("ignore")
    if not os.path.isdir(os.path.join(REF_DIR, "gptorch")):
        raise FileNotFoundError("baseline/_ref/gptorch is missing: install the reference with `python -m pip install "
                                "--no-index --no-build-isolation --no-deps --target baseline/_ref <copy of /root/reference>`")
    sys.path.insert(0, REF_DIR)
    import gptorch
    from gptorch import kernels as rk, likelihoods as rl
    from gptorch.models import GPR as RefGPR
    assert os.path.realpath(gptorch.__file__).startswith(os.path.realpath(REF_DIR))
    return rk, rl, RefGPR


class _PortModel:
    """Stand-in used ONLY when baseline/_ref is absent on the box: the oracle port of the same path (oracle/gp_oracle.py,
    torch CPU fp64).  The line then says kind = "port"."""

    def __init__(self, n):
        from oracle import gp_oracle as O
        self.O = O
        self.X, self.Y, _ = O.synth_regression(n, D_IN)

    def eval(self):
        t0 = time.perf_counter()
        loss, _ = self.O.gpr_loss_and_grads("Rbf", self.X, self.Y, np.ones(D_IN), 1.0, 0.01)
        return time.perf_counter() - t0, float(loss.item())


def _reference_model(n, mods):
    if mods is None:
        return _PortModel(n)
    rk, rl, RefGPR = mods
    X, Y, _ = synth_regression(n, D_IN)
    return RefGPR(X.numpy(), Y.numpy(), rk.Rbf(D_IN, ARD=True), likelihood=rl.Gaussian(variance=0.01))


def _reference_eval(model, cuda=False):
    if isinstance(model, _PortModel):
        return model.eval()
    for p in model.parameters():
        p.grad = None
    if cuda:
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    loss = model.loss()
    loss.backward()
    if cuda:
        torch.cuda.synchronize()
    return time.perf_counter() - t0, float(loss.item())


def _cpu_reference_modules():
    """(modules or None, kind, description): the unmodified reference when baseline/_ref travelled with the repo, else the
    oracle port."""
    try:
        return _reference_modules(), "reference", "unmodified cics-nd/gptorch (baseline/_ref, torch CPU fp64 / MKL"
    except Exception as e:  # noqa: BLE001
        sys.stderr.write("bench.py: baseline/_ref unavailable (%r) -- timing the oracle port instead\n" % (e,))
        return None, "port", "oracle/gp_oracle.py port of the reference path (baseline/_ref absent; torch CPU fp64 / MKL"


def choose_cpu_sample(n_full, evals, budget_s, mods):
    """Largest sample size whose `evals` evaluations fit the time budget, from a quick probe at N=2048."""
    avail = 64e9
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        pass
    probe = _reference_model(2048, mods)
    _reference_eval(probe)
    sec2048 = min(_reference_eval(probe)[0] for _ in range(2))
    best = 4096
    for n in (4096, 6144, 8192, 12288, 16384):
        est = sec2048 * (n / 2048.0) ** 3 * 0.8          # MKL is more efficient at the larger sizes
        if n <= n_full and est * evals <= budget_s and 9.5 * 8 * n * n <= 0.8 * avail:
            best = n
    return best


def extrapolate(sec, sample_n, n_full):
    if n_full == 32768 and sample_n in CPU_FULL_OVER_SAMPLE:
        scale = CPU_FULL_OVER_SAMPLE[sample_n]
    else:
        scale = (n_full / float(sample_n)) ** CPU_SCALING_EXPONENT
    return sec * scale, scale


def cpu_baseline(n_full, sample_n=0):
    """`cpu_baseline` of our arm's line: ONE evaluation of the unmodified reference on a bounded sample."""
    mods, kind, what = _cpu_reference_modules()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample_n = min(sample_n or choose_cpu_sample(n_full, 1, 30.0, mods), n_full)
    _reference_eval(_reference_model(1024, mods))          # warm up MKL / autograd
    sec, loss = _reference_eval(_reference_model(sample_n, mods))
    full, scale = extrapolate(sec, sample_n, n_full)
    pin = reference_pin(n_full)
    out = {"value": 1.0 / full, "unit": "evals/s", "cores": torch.get_num_threads(), "kind": kind,
           "sample": what + ", %d threads) loss+grad at N=%d, D=%d: "
                     "%.2f s measured; scaled by %.1fx to N=%d (the full-size / sample-size time ratio of the reference measured "
                     "on this pool's host where available, else (N/%d)^%.2f)" % (
                         torch.get_num_threads(), sample_n, D_IN, sec, scale, n_full, sample_n, CPU_SCALING_EXPONENT),
           "sample_n": sample_n, "sample_seconds": sec, "sample_loss": loss}
    if pin and "cpu" in pin:
        out["full_size_measured"] = {"seconds_per_eval": pin["cpu"]["seconds_best"], "threads": pin["cpu"]["threads"],
                                     "evals_per_s": 1.0 / pin["cpu"]["seconds_best"],
                                     "source": "tools/reference_box.py on this pool's GPU box host (one run, round 2), "
                                               "tests/golden/gpr_n32768_reference.json"}
    return out


def run_reference(args, rank, world):
    """--impl reference: the unmodified reference's own CPU implementation of the path, all host threads; each step is
    one loss+grad evaluation at the bounded sample size."""
    if rank != 0:
        return
    mods, kind, what = _cpu_reference_modules()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    evals = args.steps + max(args.warmup, 1)
    sample_n = min(args.cpu_sample_n or choose_cpu_sample(args.n, evals, args.cpu_budget_s, mods), args.n)
    model = _reference_model(sample_n, mods)
    for _ in range(max(args.warmup, 1)):
        _reference_eval(model)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, loss = _reference_eval(model)
    sec = (time.perf_counter() - t0) / args.steps
    full, scale = extrapolate(sec, sample_n, args.n)
    value = 1.0 / full
    pin = reference_pin(args.n)
    sample = (what + ", %d threads): model.loss() + backward() "
              "at N=%d timed %.2f s/step; value scaled by %.1fx to N=%d (the full-size / sample-size time ratio of the "
              "reference measured on this pool's host where available, else (N/%d)^%.2f)" % (
                  torch.get_num_threads(), sample_n, sec, scale, args.n, sample_n, CPU_SCALING_EXPONENT))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1000.0, "ms_per_step_is": "the measured sample step (N=%d), not the extrapolation" % sample_n,
        "ms_per_step_full_size_extrapolated": full * 1000.0,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.n, args.gpus),
        "same_config": False, "same_config_note": "the workload is the named one; each step is a bounded sample of it at "
                                                  "N=%d and `value` is an extrapolation" % sample_n,
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": sample, "sample_n": sample_n, "sample_seconds": sec, "sample_loss": loss},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if pin and "cpu" in pin:
        line["full_size_measured"] = {"seconds_per_eval": pin["cpu"]["seconds_best"], "threads": pin["cpu"]["threads"],
                                      "evals_per_s": 1.0 / pin["cpu"]["seconds_best"], "loss": pin["cpu"]["loss"],
                                      "source": "tools/reference_box.py on this pool's GPU box host (one run, round 2), "
                                                "tests/golden/gpr_n32768_reference.json"}
    print(json.dumps(line), flush=True)


def vendor_baseline(n, ours_loss):
    """The unmodified reference under model.cuda() on this GPU: torch dispatches to cuSOLVER potrf / cuBLAS trsm, dgemm
    (SURVEY 2.1 'the existing Blackwell kernel bar').  One warm-up at N=2048 (library handles), one at N, two timed."""
    try:
        mods = _reference_modules()
        warm = _reference_model(2048, mods)
        warm.cuda()
        _reference_eval(warm, cuda=True)
        del warm
        model = _reference_model(n, mods)
        model.cuda()
        torch.cuda.reset_peak_memory_stats()
        _reference_eval(model, cuda=True)
        runs = [_reference_eval(model, cuda=True) for _ in range(2)]
        sec = min(r[0] for r in runs)
        loss = runs[-1][1]
        peak = torch.cuda.max_memory_allocated() / 1e9
        del model
        torch.cuda.empty_cache()
        return {"value": 1.0 / sec, "unit": "evals/s", "seconds_per_eval": sec, "loss": loss, "peak_gb": peak,
                "loss_rel_vs_ours": abs(loss - ours_loss) / abs(ours_loss),
                "what": "unmodified cics-nd/gptorch (baseline/_ref) after model.cuda() on the same B200: torch -> cuSOLVER "
                        "potrf, cuBLAS trsm/dgemm, autograd backward; same inputs and size; host wall clock around "
                        "loss()+backward() with torch.cuda.synchronize() on both sides, best of 2 after warm-up"}
    except Exception as e:  # noqa: BLE001  (a baseline that cannot run must not take the bench down)
        torch.cuda.empty_cache()
        return {"unavailable": repr(e)[:300]}


# ------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, flag in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if v > 0.5 * (smax or 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def fp64_peak_live():
    """Measured FP64 peak on this device: best of 5 cuBLAS DGEMMs (the same way MEASURED_PEAKS.json is made)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / best / 1e9


PROBE_M, PROBE_K = 16384, 2048
PROBE_TRAFFIC_BYTES = 5.066e9   # dram__bytes_read.sum + dram__bytes_write.sum, profiles/r02_ncu_syrk_16384x2048_half_tile.txt


def dominant_launch_probe():
    """One launch shape of the dominant kernel timed on its own with CUDA events: the SYRK trailing update
    (lower tiles) m = n = 16384, k = 2048 -- the shape profiled with ncu --set full in profiles/."""
    from gptorch_b200 import _native as nv
    A = torch.randn(PROBE_M, PROBE_K, dtype=torch.float64, device="cuda")
    C = torch.randn(PROBE_M, PROBE_M, dtype=torch.float64, device="cuda")
    run = lambda: nv.gemm(nv.GEMM_NT, A, A, alpha=-1.0, beta=1.0, C=C, lower_only=True)  # noqa: E731
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    times = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run(); e1.record(); torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    tiles = (PROBE_M // 128) * (PROBE_M // 128 + 1) // 2
    flop = 2.0 * tiles * 128 * 128 * PROBE_K
    del A, C
    torch.cuda.empty_cache()
    return {"shape": "syrk lower m=n=%d k=%d (%d tiles of 128x128; C is 2.1 GB > L2)" % (PROBE_M, PROBE_K, tiles),
            "ms": ms, "flop": flop, "tflops": flop / ms / 1e9}


def build_model(n, device):
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import GPR
    X, Y, _ = synth_regression(n, D_IN)
    model = GPR(X.numpy(), Y.numpy(), kernels.Rbf(D_IN, ARD=True), likelihood=likelihoods.Gaussian(variance=0.01))
    return model, X, Y


def one_eval(model):
    for p in model.parameters():
        p.grad = None
    loss = model.loss()
    loss.backward()
    return loss


def dump_outputs(out_dir, arrays):
    """Write every array as out_dir/<name>.npy in float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def check_parity(n, loss_value, grads, fatal=True):
    """Loss (<= 1e-9) and gradients (<= 1e-7) of the timed evaluation against the unmodified reference's values at the
    named size; raises if the fast path has drifted -- a fast kernel whose results differ is not done.  (fatal=False:
    report `within_tolerance` instead, used for the experimental int8-sliced engine.)"""
    pin = reference_pin(n)
    if pin is None:
        return {"loss_pin": None, "parity": "no reference pin for N=%d" % n}
    out = {"source": "tests/golden/gpr_n32768_reference.json (unmodified reference on this pool's box: host CPU/MKL and "
                     "model.cuda())"}
    for arm in ("cpu", "cuda"):
        ref = pin.get(arm)
        if not ref:
            continue
        rel_loss = abs(loss_value - ref["loss"]) / abs(ref["loss"])
        rel_grad = max(float(np.abs(np.asarray(grads[k]) - np.asarray(v)).max() / np.abs(np.asarray(v)).max())
                       for k, v in ref["grads"].items())
        out["loss_pin_" + arm] = ref["loss"]
        out["loss_rel_vs_reference_" + arm] = rel_loss
        out["grad_rel_vs_reference_" + arm] = rel_grad
        if not fatal:
            out["within_tolerance"] = out.get("within_tolerance", True) and rel_loss <= 1e-9 and rel_grad <= 1e-7
        elif rel_loss > 1e-9 or rel_grad > 1e-7:
            raise SystemExit("bench.py: PARITY FAILURE against the reference (%s arm): loss rel %.3e, gradient rel %.3e"
                             % (arm, rel_loss, rel_grad))
    out["loss_pin"] = pin["cpu"]["loss"] if "cpu" in pin else pin["cuda"]["loss"]
    return out


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from gptorch_b200 import _native as nv
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    n = args.n
    model, X, Y = build_model(n, device)
    params = [p for p in model.parameters() if p.requires_grad]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing -----------------------------------------------------------
    for _ in range(args.warmup):
        loss = one_eval(model)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    timer = nv.PhaseTimer()
    nv.install_timer(timer)
    nv.reset_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = one_eval(model)
    e1.record()
    barrier()
    launches = nv.launch_count()
    nv.install_timer(None)
    ms = e0.elapsed_time(e1)
    phases = timer.totals_ms()
    clocks = sampler.stop() if rank == 0 else None
    loss_value = float(loss.item())
    grads = {"kernel.variance": model.kernel.variance.grad.cpu().numpy(),
             "kernel.length_scales": model.kernel.length_scales.grad.cpu().numpy(),
             "likelihood.variance": model.likelihood.variance.grad.cpu().numpy()}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss.detach().cpu().numpy(),
                                         **{name + ".grad": g for name, g in grads.items()}})
    parity = check_parity(n, loss_value, grads)

    # ---------------- end-to-end through the public API with host inputs, all K steps ------------------------
    x_host = X.clone().pin_memory()
    y_host = Y.clone().pin_memory()
    one_eval(model)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.X.copy_(x_host, non_blocking=True)
        model.Y.copy_(y_host, non_blocking=True)
        loss = one_eval(model)
        host_loss = loss.detach().cpu()
        host_grads = [p.grad.detach().cpu() for p in params]
    torch.cuda.synchronize()
    e2e_sec = time.perf_counter() - t0
    h2d = (x_host.numel() + y_host.numel()) * 8
    d2h = (host_loss.numel() + sum(g.numel() for g in host_grads)) * 8

    # ---------------- EXPERIMENTAL engine, reported beside the headline (never part of `value`) -----------------
    int8_sliced = None
    if world == 1 and not args.no_int8_sliced and n >= 8192:
        int8_sliced = {"what": "the same loss+grad with the O(N^3) products of gpb_potrf_lower / gpb_potri_lower on the INT8 "
                               "tensor path: FP64 operands cut into 7-bit slices by this library's split kernel, slice products "
                               "by cuBLASLt int8 GEMMs (library calls) over a concatenated k, fp64 recombination by this "
                               "library's kernel (csrc/gpb_ozaki.cu; off by default: GPB_OZAKI / gpb_ozaki_config). Everything "
                               "else -- and `value`, `e2e`, `roofline` above -- is the hand-written FP64 DMMA path.",
                       "runs": {}}
        def grads_now():
            return {"kernel.variance": model.kernel.variance.grad.cpu().numpy(),
                    "kernel.length_scales": model.kernel.length_scales.grad.cpu().numpy(),
                    "likelihood.variance": model.likelihood.variance.grad.cpu().numpy()}
        try:
            for slices in (8, 7):
                nv.ozaki_config(slices)
                for _ in range(2):
                    one_eval(model)
                timer2 = nv.PhaseTimer()
                nv.install_timer(timer2)
                torch.cuda.synchronize()
                k_steps = args.steps
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                for _ in range(k_steps):
                    loss8 = one_eval(model)
                f1.record()
                torch.cuda.synchronize()
                nv.install_timer(None)
                ms8 = f0.elapsed_time(f1) / k_steps
                ph8 = timer2.totals_ms()
                int8_sliced["runs"]["slices_%d" % slices] = {
                    "ms_per_step": ms8, "evals_per_s": 1000.0 / ms8, "speedup_vs_dmma": (ms / args.steps) / ms8,
                    "steps": k_steps, "phases_ms_per_step": {k: v / k_steps for k, v in sorted(ph8.items())},
                    "fp64_equivalent_tflops_potrf_potri": float(n) ** 3 / ((ph8.get("potrf", 0) + ph8.get("potri", 0)) / k_steps) / 1e9,
                    "loss": float(loss8.item()),
                    "parity": check_parity(n, float(loss8.item()), grads_now(), fatal=False)}
        except Exception as exc:    # the experimental engine must never take the bench line down
            int8_sliced["error"] = "%s: %s" % (type(exc).__name__, exc)
        finally:
            nv.install_timer(None)
            nv.ozaki_config(0)

    t = torch.tensor([ms, e2e_sec * 1000.0], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = t[0].item(), t[1].item()
    del model
    torch.cuda.empty_cache()

    # ---------------- the configurations that shard (all ranks take part) ------------------------------------
    sharded = None
    if not args.no_sharded and n == 32768:
        import bench_sharded
        sharded = bench_sharded.run(rank, world, device, ms_max / args.steps, parity.get("loss_pin"), args.steps)
    if rank != 0:
        return

    steps = args.steps
    value = world * steps / (ms_max / 1000.0)
    e2e_value = world * steps / (e2e_ms_max / 1000.0)
    peak_issue = nv.dmma_issue_peak_tflops()
    peak_cublas = fp64_peak_live()
    potrf_ms = phases.get("potrf", 0.0) / steps
    potri_ms = phases.get("potri", 0.0) / steps
    n3 = float(n) ** 3
    chol_tflops = n3 / 3.0 / potrf_ms / 1e9 if potrf_ms else None
    o3_tflops = n3 / (potrf_ms + potri_ms) / 1e9 if (potrf_ms + potri_ms) else None
    probe = dominant_launch_probe()
    line = {
        "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(n, world),
        "loss": loss_value, "parity": parity,
        "chol_tflops": chol_tflops,
        "phases_ms_per_step": {k: v / steps for k, v in sorted(phases.items())},
        "roofline": {"bound": "tensor", "achieved": o3_tflops, "peak": peak_issue, "unit": "TFLOP/s",
                     "frac": (o3_tflops / peak_issue) if o3_tflops else None,
                     "traffic": PROBE_TRAFFIC_BYTES,
                     "kernel": "gemm_dmma_kernel (FP64 DMMA.8x8x4 fed by TMA; 128x64 half tiles, two CTAs per SM) -- > 95 % of "
                               "gpb_potrf_lower + gpb_potri_lower",
                     "algorithmic": "achieved = N^3 flop per eval (potrf N^3/3 + potri 2N^3/3) / CUDA-event time of those two "
                                    "phases inside the timed steps (all their launches, including the latency-bound ones)",
                     "peak_source": "measured live: FP64 tensor-pipe issue ceiling (gpb_dmma_issue_probe: independent "
                                    "DMMA.8x8x4 chains from registers, 2 CTAs x 16 warps per SM); MEASURED_PEAKS.json has no "
                                    "FP64 entry and the profiling guide states no FP64 fallback",
                     "peak_cublas_dgemm_live": peak_cublas,
                     "frac_vs_cublas_dgemm_live": (o3_tflops / peak_cublas) if o3_tflops else None,
                     "chol_frac": (chol_tflops / peak_issue) if chol_tflops else None,
                     "launch_probe": probe,
                     "traffic_note": "dram__bytes_read+write of ONE launch of the probe shape from ncu --set full "
                                     "(profiles/r02_ncu_syrk_16384x2048_half_tile.txt: DMMA sub-pipe 96.5 % active); "
                                     "algorithmic bytes of that launch: 2.43e9"},
        "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if int8_sliced is not None:
        line["int8_sliced_experimental"] = int8_sliced
    if sharded is not None:
        line["sharded"] = sharded
    if world == 1 and not args.no_vendor_baseline:
        line["vendor_baseline"] = vendor_baseline(n, loss_value)
    if not args.no_cpu_baseline and world == 1:     # reported on rank 0 of the single-GPU run only
        line["cpu_baseline"] = cpu_baseline(n, args.cpu_sample_n)
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (gptorch_b200 has no CPU path); use --impl reference for the CPU arm")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
