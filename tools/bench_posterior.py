"""Cost of a differentiable prediction: ms per mean + variance + x* gradient through GPR.posterior() against
GPR.predict_f with autograd (which refactorises on every call), the one-time cost of posterior(), peak memory, and the
kernel time of gpb_pred_gx with FLOP/s and bytes/s from shape-derived counts.

Cases: GPR Rbf-ARD D = 8, N in {8192, 32768}, n* in {1, 64, 1024}.  The two paths alternate inside one process (CUDA
events around each prediction + backward, after a warm-up of both), so drift of the shared host affects both alike.
Ky^-1 (N^2 doubles) is larger than the L2 cache at both N, so every call reads it from HBM.  Prints one JSON line per
case plus the device name and power limit it ran on.

    python tools/bench_posterior.py [--reps 10] [--model-reps 3] [--out profiles/r04_posterior.json]
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

KB_COLS, DC = 128, 8     # gpb_pred_gx: test rows per CTA, feature chunk for D <= 8


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = "unavailable (%r)" % (e,)
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def make_model(n, d):
    from oracle import gp_oracle as O
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import GPR
    X, Y, _ = O.synth_regression(n, d)
    ell = 0.5 + 0.1 * np.arange(d)
    return GPR(X.numpy(), Y.numpy(), kernels.Rbf(d, ARD=True, length_scales=ell.copy(), variance=1.3),
               likelihood=likelihoods.Gaussian(variance=0.02))


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def predict_step(source, xs):
    x = xs.detach().clone().requires_grad_(True)
    mean, var = source.predict_f(x)
    # weighted sums: materialised upstream gradients (predict_f's GEMM backward rejects the stride-0 1 x 1 gradient
    # that mean.sum() hands it at n* = 1)
    (mean * torch.ones_like(mean) + var * torch.ones_like(var)).sum().backward()
    return x.grad


def peak_of(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def pred_gx_counts(ns, n, d, dy):
    """Shape-derived work of one gpb_pred_gx launch: per (test, training) pair the distance (3 D), W (2 dy + 2) and the
    feature accumulation (3 D) -- the kernel function's exp is not counted; bytes of Q, X and a as each CTA reads them,
    plus x*, g_mean, g_var and the output."""
    ctas_m, ctas_d = (ns + KB_COLS - 1) // KB_COLS, (d + DC - 1) // DC
    flop = ns * n * (6 * d + 2 * dy + 2)
    byts = 8 * (ctas_d * ns * n + ctas_m * ctas_d * n * (d + dy) + ns * (2 * d + dy + 1))
    return flop, byts


def kernel_time(post, xs, launches):
    """CUDA-event time of gpb_pred_gx alone, averaged over `launches` back-to-back launches on the saved forward."""
    from gptorch_b200 import _native as nv
    kind, X, a = post._kind, post.X, post.a
    ell, s2 = post.kernel.length_scales.transform(), post.kernel.variance.transform()
    Ks = nv.kern_fwd(kind, xs, X, ell, s2)
    Q = nv.gemm(nv.GEMM_NN, Ks, post.Kinv)
    del Ks
    gm = torch.ones(xs.shape[0], a.shape[1], dtype=torch.float64, device=xs.device)
    gv = torch.ones(xs.shape[0], dtype=torch.float64, device=xs.device)
    nv.pred_gx(kind, xs, X, ell, s2, a, gm, gv, Q)
    ms, _ = timed(lambda: [nv.pred_gx(kind, xs, X, ell, s2, a, gm, gv, Q) for _ in range(launches)])
    return ms / launches


def measure_n(n, d, sizes, reps, model_reps):
    model = make_model(n, d)
    model.posterior()                                     # warm-up of every shape posterior() launches
    torch.cuda.synchronize()
    post_ms = []
    post = None
    for _ in range(2):
        post = None
        torch.cuda.empty_cache()
        ms, post = timed(model.posterior)
        post_ms.append(ms)
    post_peak = peak_of(model.posterior)
    g = torch.Generator().manual_seed(7)
    out = []
    for ns in sizes:
        xs = (3.0 * torch.rand(ns, d, generator=g, dtype=torch.float64) - 1.0).cuda()
        for src in (post, model):
            predict_step(src, xs)
        model.zero_grad(set_to_none=True)
        t_post, t_model = [], []
        for r in range(max(reps, model_reps)):
            if r < reps:
                t_post.append(timed(lambda: predict_step(post, xs))[0])
            if r < model_reps:
                t_model.append(timed(lambda: predict_step(model, xs))[0])
        model.zero_grad(set_to_none=True)
        peak_post = peak_of(lambda: predict_step(post, xs))
        peak_model = peak_of(lambda: predict_step(model, xs))
        model.zero_grad(set_to_none=True)
        k_ms = kernel_time(post, xs, 20)
        flop, byts = pred_gx_counts(ns, n, d, 1)
        mp, mm = float(np.median(t_post)), float(np.median(t_model))
        r = {"case": "GPR Rbf-ARD D=%d N=%d n*=%d" % (d, n, ns),
             "ms_posterior": t_post, "ms_predict_f_autograd": t_model,
             "median_ms_posterior": mp, "median_ms_predict_f_autograd": mm, "speedup": mm / mp,
             "posterior_build_ms": post_ms, "posterior_build_peak_bytes": post_peak,
             "posterior_cache_bytes": int(post.Kinv.untyped_storage().nbytes()),
             "peak_bytes_posterior_call": peak_post, "peak_bytes_predict_f_call": peak_model,
             "pred_gx_kernel_ms": k_ms, "pred_gx_flop": flop, "pred_gx_bytes": byts,
             "pred_gx_gflops": flop / k_ms / 1e6, "pred_gx_gbytes_per_s": byts / k_ms / 1e6}
        print(json.dumps(r), flush=True)
        out.append(r)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="timed calls through the posterior per case")
    ap.add_argument("--model-reps", type=int, default=3, help="timed calls through predict_f per case")
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a run-through of the script, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_posterior.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    info = device_info()
    print(json.dumps(info), flush=True)
    results = [info]
    ns_sizes = (1, 64, 1024)
    for n in ((1000, 2000) if args.small else (8192, 32768)):
        results += measure_n(n, 8, ns_sizes, args.reps, args.model_reps)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
