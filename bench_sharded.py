"""The configurations of BASELINE.json that SHARD (SURVEY 8e), measured inside bench.py's run and printed in its JSON
line as the `sharded` block.  One process per GPU (bench.py owns the process group); every number is CUDA-event timed
between barriers and reported as the max over ranks; every result is cross-checked against a single-GPU evaluation
or a reference pin.

  vfe      configs[2]  VFE Rbf-ARD N=1e7, D=16, M=1024: rows split over the ranks (STRONG scaling of the same data set),
                       one all-reduce of the M x M statistics forward, one of the streamed gradients backward.
  svgp     configs[3]  SVGP Matern52-ARD M=2048, D=32, minibatch 65536 per GPU (WEAK scaling, data parallel),
                       one all-reduce of the flat gradient per step.
  dist_gpr configs[1]/[4]  exact GPR through the block-column-cyclic distributed Cholesky + inverse + gradient:
                       N=32768 strong-scaled against the single-GPU fused node; N=131072 (configs[4]) on 8 GPUs.
"""
import time

import numpy as np
import torch
import torch.distributed as dist

FP64_PEAK_TFLOPS = 37.05          # DMMA issue ceiling of one B200 (profiles/r01_fp64_peak.txt; bench.py re-measures it)
VFE_N, VFE_D, VFE_M, VFE_SHARDS = 10_000_000, 16, 1024, 8
SVGP_B, SVGP_M, SVGP_D, SVGP_ROWS = 65536, 2048, 32, 262144
C5_N = 131072
C5_LOSS_R01 = -113952.01193680815   # profiles/r01_multigpu.json (8-rank runs of round 1 with 512/1024/2048-column panels)


def _sync(world):
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _timed(fn, steps, world, device):
    """ms per call of fn(): CUDA events on the current stream between barriers, max over ranks."""
    _sync(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for _ in range(steps):
        out = fn()
    e1.record()
    _sync(world)
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item(), out


def _allreduce_ms(numel, world, device, reps=10):
    """Cost of one all-reduce of `numel` doubles on this group (CUDA events, max over ranks); 0 for one rank."""
    if world == 1:
        return 0.0
    buf = torch.zeros(numel, dtype=torch.float64, device=device)
    for _ in range(3):
        dist.all_reduce(buf)
    ms, _ = _timed(lambda: dist.all_reduce(buf), reps, world, device)
    return ms


# ------------------------------------------------------------------------------------------------------------
# VFE, configs[2]
# ------------------------------------------------------------------------------------------------------------
def _vfe_rows(shards, w):
    xs, ys = [], []
    for s in shards:
        g = torch.Generator().manual_seed(1000 + s)
        X = torch.rand(VFE_N // VFE_SHARDS, VFE_D, generator=g, dtype=torch.float64)
        xs.append(X)
        ys.append(torch.sin(X @ w) + 0.1 * torch.randn(X.shape[0], 1, generator=g, dtype=torch.float64))
    return torch.cat(xs), torch.cat(ys)


def _vfe_model(shards, distributed):
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import VFE
    g = torch.Generator().manual_seed(1234)
    w = torch.randn(VFE_D, 1, generator=g, dtype=torch.float64)
    Z = torch.rand(VFE_M, VFE_D, generator=g, dtype=torch.float64)
    X, Y = _vfe_rows(shards, w)
    model = VFE(X, Y, kernels.Rbf(VFE_D, ARD=True), inducing_points=Z.numpy(), likelihood=likelihoods.Gaussian(variance=0.01))
    if distributed:
        model.distribute()
    return model


def _step(model, post=None):
    for p in model.parameters():
        p.grad = None
    loss = model.loss()
    loss.sum().backward()
    if post is not None:
        post(model)
    return loss.detach()


def bench_vfe(rank, world, device, steps):
    per = VFE_SHARDS // world
    model = _vfe_model(range(rank * per, (rank + 1) * per), world > 1)
    _step(model)
    ms, loss = _timed(lambda: _step(model), steps, world, device)
    grads = torch.cat([model.kernel.length_scales.grad.reshape(-1), model.kernel.variance.grad.reshape(-1),
                       model.likelihood.variance.grad.reshape(-1), model.Z.grad.reshape(-1)]).clone()
    flop = 3.0 * VFE_N * VFE_M ** 2 + 6.0 * VFE_N * VFE_M * VFE_D            # SURVEY 8d algorithmic count
    cond = getattr(model, "last_kuu_condition", None)
    from gptorch_b200 import settings
    phi = cond is not None and cond <= settings.vfe_phi_cond_max
    out = {"workload": "VFE Rbf-ARD fp64 N=%d D=%d M=%d loss+grad (configs[2]), rows sharded over %d rank(s)"
                       % (VFE_N, VFE_D, VFE_M, world),
           "scaling": "strong", "steps": steps, "ms_per_eval": ms, "evals_per_s": 1000.0 / ms,
           "rows_per_s": VFE_N / (ms / 1000.0),
           "loss": float(loss.item()),
           "form": ("Phi form, 3 N M^2 + 6 N M D flop executed (condition-gated: estimated cond_2(Kuu) = %.3g <= %.3g)"
                    % (cond, settings.vfe_phi_cond_max)) if phi else
                   "reference order of operations, 5 N M^2 flop executed (estimated cond_2(Kuu) = %s)" % cond,
           "flop_counted": "3 N M^2 + 6 N M D (SURVEY 8d algorithmic count)",
           "algorithmic_tflops_per_gpu": flop / world / (ms / 1000.0) / 1e12,
           "frac_of_fp64_peak": flop / world / (ms / 1000.0) / 1e12 / FP64_PEAK_TFLOPS,
           "collectives": "all_reduce(M*M + M*dy + 2 doubles) forward, all_reduce(D + 1 + M*D doubles) backward",
           "allreduce_ms_fwd": _allreduce_ms(VFE_M * VFE_M + VFE_M + 2, world, device),
           "allreduce_ms_bwd": _allreduce_ms(VFE_D + 1 + VFE_M * VFE_D, world, device)}
    del model
    torch.cuda.empty_cache()
    if world > 1:
        # the SAME data set on ONE GPU (rank 0 alone): the strong-scaling baseline and the cross-check
        flat = torch.zeros(grads.numel() + 2, dtype=torch.float64, device=device)
        if rank == 0:
            single = _vfe_model(range(VFE_SHARDS), False)
            _step(single)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            l1 = _step(single)
            e1.record()
            torch.cuda.synchronize()
            g1 = torch.cat([single.kernel.length_scales.grad.reshape(-1), single.kernel.variance.grad.reshape(-1),
                            single.likelihood.variance.grad.reshape(-1), single.Z.grad.reshape(-1)])
            flat[0], flat[1], flat[2:] = e0.elapsed_time(e1), l1.item(), g1
            del single
            torch.cuda.empty_cache()
        dist.broadcast(flat, src=0)
        single_ms, single_loss, g1 = flat[0].item(), flat[1].item(), flat[2:]
        out.update({"single_gpu_ms_per_eval": single_ms, "speedup_vs_single_gpu": single_ms / ms,
                    "strong_scaling_efficiency": single_ms / ms / world,
                    "loss_rel_vs_single_gpu": abs(out["loss"] - single_loss) / abs(single_loss),
                    "grad_rel_vs_single_gpu": float((grads - g1).abs().max() / g1.abs().max())})
    return out


# ------------------------------------------------------------------------------------------------------------
# SVGP, configs[3]
# ------------------------------------------------------------------------------------------------------------
def bench_svgp(rank, world, device, steps):
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.dist import allreduce_grads
    from gptorch_b200.models import SVGP
    g = torch.Generator().manual_seed(1234)
    w = torch.randn(SVGP_D, 1, generator=g, dtype=torch.float64)
    Z = torch.rand(SVGP_M, SVGP_D, generator=g, dtype=torch.float64)
    gr = torch.Generator().manual_seed(2000 + rank)
    X = torch.rand(SVGP_ROWS, SVGP_D, generator=gr, dtype=torch.float64)
    Y = torch.sin(X @ w) + 0.1 * torch.randn(SVGP_ROWS, 1, generator=gr, dtype=torch.float64)
    np.random.seed(rank)
    model = SVGP(X, Y, kernels.Matern52(SVGP_D, ARD=True, length_scales=2.0 * np.ones(SVGP_D)), inducing_points=Z.numpy(),
                 likelihood=likelihoods.Gaussian(variance=0.01), batch_size=SVGP_B)
    if world > 1:
        model.distribute()          # broadcasts rank 0's parameters (q(u) is initialised from the local shard)
    post = (lambda m: allreduce_grads(m)) if world > 1 else None
    _step(model, post)
    ms, loss = _timed(lambda: _step(model, post), steps, world, device)
    nparam = sum(p.numel() for p in model.parameters() if p.requires_grad)
    from gptorch_b200 import settings
    cond = getattr(model, "last_kuu_condition", None)
    quad = cond is not None and cond <= settings.vfe_phi_cond_max
    # flop actually executed per step and GPU: the quadratic form needs 3 B M^2 (one panel product 2 B M^2, one Gram
    # product B M^2) + 4 B M D, the reference order 6 B M^2 (SURVEY 8d's ~1.7e12); both + O(M^3) replicated algebra
    flop = (3.0 if quad else 6.0) * SVGP_B * SVGP_M ** 2 + 4.0 * SVGP_B * SVGP_M * SVGP_D + 20.0 * SVGP_M ** 3
    # replicas must stay identical: same parameters in, all-reduced gradients out
    chk = model.induced_output_mean.grad.abs().sum().reshape(1).clone()
    lo, hi = chk.clone(), chk.clone()
    if world > 1:
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    out = {"workload": "SVGP Matern52-ARD fp64 M=%d D=%d, minibatch %d per GPU x %d rank(s) (configs[3]; each rank's "
                       "shard of %d rows is resident in HBM)" % (SVGP_M, SVGP_D, SVGP_B, world, SVGP_ROWS),
           "scaling": "weak", "steps": steps, "ms_per_step": ms, "points_per_s": world * SVGP_B / (ms / 1000.0),
           "loss_rank0": float(loss.item()),
           "form": ("quadratic form (M x M algebra first), 3 B M^2 flop executed (condition-gated: estimated cond_2(Kuu) = "
                    "%.3g <= %.3g)" % (cond, settings.vfe_phi_cond_max)) if quad else
                   "reference order of operations, 6 B M^2 flop executed (estimated cond_2(Kuu) = %s)" % cond,
           "flop_counted": "executed: %.3g per step and GPU" % flop,
           "algorithmic_tflops_per_gpu": flop / (ms / 1000.0) / 1e12,
           "frac_of_fp64_peak": flop / (ms / 1000.0) / 1e12 / FP64_PEAK_TFLOPS,
           "collectives": "all_reduce(flat gradient, %d doubles = %.1f MB) per step" % (nparam, nparam * 8 / 1e6),
           "allreduce_ms": _allreduce_ms(nparam, world, device),
           "replicas_agree": bool((hi - lo).item() <= 1e-12 * abs(hi.item()))}
    del model
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------------
# distributed exact GPR, configs[1] strong-scaled and configs[4]
# ------------------------------------------------------------------------------------------------------------
def bench_dist_gpr(rank, world, device, n, steps, single_gpu_ms=None, loss_pin=None, warm=True):
    from bench import synth_regression
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import DistributedGPR
    from gptorch_b200.models import dist_gpr as dg
    X, Y, _ = synth_regression(n, 8)
    model = DistributedGPR(X.numpy(), Y.numpy(), kernels.Rbf(8, ARD=True), likelihood=likelihoods.Gaussian(variance=0.01),
                           panel=1024)
    if warm:
        _step(model)
    from gptorch_b200 import _native as nv
    dg.WAIT_LOG = []
    timer = nv.PhaseTimer()
    nv.install_timer(timer)
    ms, loss = _timed(lambda: _step(model), steps, world, device)
    nv.install_timer(None)
    stages = timer.totals_ms()
    waits, dg.WAIT_LOG = dg.WAIT_LOG, None
    wait_ms = [a.elapsed_time(b) for a, b in waits]
    wait = torch.tensor([sum(wait_ms) / steps], dtype=torch.float64, device=device)       # per evaluation
    if world > 1:
        dist.all_reduce(wait, op=dist.ReduceOp.MAX)
    panels = (n + 1023) // 1024
    out = {"workload": "exact GPR Rbf-ARD fp64 N=%d D=8 loss+grad, block-column-cyclic Cholesky + inverse + gradient over "
                       "%d rank(s), 1024-column panels" % (n, world),
           "scaling": "strong", "steps": steps, "ms_per_eval": ms, "loss": float(loss.item()),
           "tflops_aggregate": float(n) ** 3 / (ms / 1000.0) / 1e12,
           "frac_of_aggregate_fp64_peak": float(n) ** 3 / (ms / 1000.0) / 1e12 / (world * FP64_PEAK_TFLOPS),
           "collectives": "ncclBroadcast of each factored panel ((N - c) x 1024 doubles) in 3 sweeps (L, T = L^-1, Kinv), "
                          "all_reduce of a (N doubles) and of D + 2 gradient doubles",
           "stage_ms_rank0": {k: v / steps for k, v in sorted(stages.items()) if k.startswith("dist_")},
           "stage_note": "dist_potrf / dist_trtri / dist_lauum are N^3/3 flop each, spread over the ranks; per evaluation",
           "panel_wait_ms_total_max_rank": wait.item(), "panel_waits": len(wait_ms) // steps,
           "panel_wait_ms_per_panel": wait.item() / max(3 * panels, 1),
           "max_mem_gb": torch.cuda.max_memory_allocated() / 1e9}
    if single_gpu_ms:
        out["single_gpu_ms_per_eval"] = single_gpu_ms
        out["speedup_vs_single_gpu"] = single_gpu_ms / ms
        out["strong_scaling_efficiency"] = single_gpu_ms / ms / world
    if loss_pin is not None:
        out["loss_rel_vs_pin"] = abs(out["loss"] - loss_pin) / abs(loss_pin)
    del model
    torch.cuda.empty_cache()
    return out


def run(rank, world, device, single_gpu_ms, loss_pin, steps, budget_s=240.0):
    """The `sharded` block of bench.py's JSON line; every configuration times `steps` steps (bench.py --steps)."""
    t0 = time.perf_counter()
    out = {"n_gpus": world}
    out["vfe"] = bench_vfe(rank, world, device, steps)
    out["svgp"] = bench_svgp(rank, world, device, steps)
    if world > 1:
        out["dist_gpr_n32768"] = bench_dist_gpr(rank, world, device, 32768, steps, single_gpu_ms, loss_pin)
    if world >= 8 and time.perf_counter() - t0 < budget_s:
        out["dist_gpr_n131072"] = bench_dist_gpr(rank, world, device, C5_N, steps, None, C5_LOSS_R01, warm=False)
    out["seconds"] = time.perf_counter() - t0
    return out
