"""Cost of the input gradient: ms per loss + grad and peak memory with x.requires_grad False vs True.

Cases: GPR Rbf-ARD D = 8 at N = 8192 and 32768 (fused stationary node), VFE Matern52-ARD at N = 1.25e6, M = 1024,
D = 16 on one GPU (the Phi form that settings.vfe_phi_form = "auto" picks there).  The two settings alternate inside
one process (CUDA events around each loss + backward, after a warm-up of both), so drift of the shared host affects
both alike.  Prints one JSON line per case plus the device name and power limit it ran on.

    python tools/bench_input_grad.py [--reps 5] [--out profiles/r03_input_grad.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = "unavailable (%r)" % (e,)
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def gpr_case(n, d):
    from oracle import gp_oracle as O
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import GPR
    X, Y, _ = O.synth_regression(n, d)
    ell = 0.5 + 0.1 * np.arange(d)
    model = GPR(X.numpy(), Y.numpy(), kernels.Rbf(d, ARD=True, length_scales=ell.copy(), variance=1.3),
                likelihood=likelihoods.Gaussian(variance=0.02))
    return model, model.X.detach().clone().cuda()


def vfe_case(n, m, d):
    from oracle import gp_oracle as O
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import VFE
    g = torch.Generator().manual_seed(1234)
    X = torch.rand(n, d, generator=g, dtype=torch.float64)
    w = torch.randn(d, 1, generator=g, dtype=torch.float64)
    Y = torch.sin(X @ w) + 0.1 * torch.randn(n, 1, generator=g, dtype=torch.float64)
    Z = O.synth_inducing(X, m, g)
    ell = 0.5 + 0.1 * np.arange(d)
    model = VFE(X.numpy(), Y.numpy(), kernels.Matern52(d, ARD=True, length_scales=ell.copy(), variance=1.3),
                inducing_points=Z.numpy(), likelihood=likelihoods.Gaussian(variance=0.05))
    return model, model.X.detach().clone().cuda()


def step(model, x0, need_x):
    model.zero_grad(set_to_none=True)
    x = x0.detach().requires_grad_(need_x)
    loss = -model.log_likelihood(x=x)
    loss.sum().backward()
    return x.grad


def measure(name, model, x0, reps):
    for need_x in (False, True):            # warm-up of both shapes of the backward pass
        step(model, x0, need_x)
    torch.cuda.synchronize()
    times = {False: [], True: []}
    peak = {}
    for need_x in (False, True):
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        step(model, x0, need_x)
        torch.cuda.synchronize()
        peak[need_x] = torch.cuda.max_memory_allocated()
    for _ in range(reps):
        for need_x in (False, True):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step(model, x0, need_x)
            b.record()
            torch.cuda.synchronize()
            times[need_x].append(a.elapsed_time(b))
    med = {k: float(np.median(v)) for k, v in times.items()}
    return {"case": name, "reps": reps,
            "ms_no_x_grad": times[False], "ms_x_grad": times[True],
            "median_ms_no_x_grad": med[False], "median_ms_x_grad": med[True],
            "median_extra_ms": med[True] - med[False],
            "peak_bytes_no_x_grad": peak[False], "peak_bytes_x_grad": peak[True],
            "extra_peak_bytes": peak[True] - peak[False]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a run-through of the script, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_input_grad.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    info = device_info()
    print(json.dumps(info), flush=True)
    results = [info]
    gpr_sizes = (512, 1000) if args.small else (8192, 32768)
    vfe_size = (20000, 128, 16) if args.small else (1250000, 1024, 16)
    for n in gpr_sizes:
        model, x0 = gpr_case(n, 8)
        r = measure("GPR Rbf-ARD N=%d D=8" % n, model, x0, args.reps)
        print(json.dumps(r), flush=True)
        results.append(r)
        del model, x0
    n, m, d = vfe_size
    model, x0 = vfe_case(n, m, d)
    r = measure("VFE Matern52-ARD N=%d M=%d D=%d" % (n, m, d), model, x0, args.reps)
    print(json.dumps(r), flush=True)
    results.append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
