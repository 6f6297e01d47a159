"""Times the three engines of the O(N^3) products side by side in one process, alternating them shape by shape: the FP64
DMMA engine, the library int8-sliced engine (cuBLASLt products, gpb_ozaki_config) and the fused tcgen05 int8-sliced
kernel (gpb_i8mma_config, the default; its inverse runs at INVERSE_SLICES in 32-column tiles, whatever --slices says).
Shapes: the SYRK-shaped trailing update C -= P P^T (lower blocks, m = 30720, k = 2048) and gpb_potrf_lower /
gpb_potri_lower at N = 16384 and 32768.  For each: time (median of the repetitions), int8
TOP/s of every shape on the sliced engines (the whole shape's FP64-equivalent flops times the S(S+1)/2 class products;
for potrf and potri this counts the DMMA panels as if sliced, so it slightly overstates the products' rate),
FP64-equivalent TFLOP/s, peak device memory, plus the card's name, power limit and maximum SM clock.

    python tools/bench_ozaki_mma.py [--reps R] [--slices S] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from gptorch_b200 import _native as nv  # noqa: E402

ENGINES = ("dmma", "library", "native")
INVERSE_SLICES = 9          # the fused engine's slice count for gpb_potri_lower's products (csrc/gpb_ozaki.cuh)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def use(engine, slices):
    nv.ozaki_config(slices if engine == "library" else 0)
    nv.i8mma_config(slices if engine == "native" else 0)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2], ts


def device_used_bytes():
    """Device memory in use right after an engine ran: the operands plus the engine's own workspace, which it keeps
    (cudaMalloc outside torch's allocator) until it is switched off."""
    free, total = torch.cuda.mem_get_info()
    return total - free


def syrk_case(m, k, slices, reps):
    g = torch.Generator().manual_seed(5)
    X = torch.rand(m, 8, generator=g, dtype=torch.float64)
    P = torch.exp(-0.5 * torch.cdist(X, X[:k]).pow(2)).cuda()
    C = torch.zeros(m, m, dtype=torch.float64, device="cuda")
    fp64_flop = float(m) * (m + 128) * k                          # lower 128-blocks of 2 m^2 k / 2
    res = {}
    for eng in ENGINES:
        use(eng, slices)
        if eng == "dmma":
            fn = lambda: nv.gemm(nv.GEMM_NT, P, P, alpha=-1.0, beta=1.0, C=C, lower_only=True)  # noqa: E731
        else:
            fn = lambda: nv.gemm_ozaki_nt(P, None, slices=slices, alpha=-1.0, beta=1.0, C=C, lower_only=True)  # noqa: E731
        ms, ts = timed(fn, reps)
        r = {"ms": ms, "all_ms": ts, "fp64_equiv_tflops": fp64_flop / ms * 1e-9, "device_used_bytes": device_used_bytes()}
        if eng != "dmma":
            r["int8_tops"] = fp64_flop * slices * (slices + 1) / 2 / ms * 1e-9
        res[eng] = r
        use("dmma", slices)                # returns the sliced engines' workspaces before the next engine runs
    return res


def factor_case(n, slices, reps):
    g = torch.Generator().manual_seed(6)
    X = torch.rand(n, 8, generator=g, dtype=torch.float64).cuda()
    ell = torch.ones(8, dtype=torch.float64, device="cuda")
    s2 = torch.ones(1, dtype=torch.float64, device="cuda")
    noise = torch.full((1,), 0.01, dtype=torch.float64, device="cuda")
    buf, ld = nv._aligned_empty(n, n, X.device)
    res = {}
    for eng in ENGINES:
        use(eng, slices)
        state = {}

        def potrf():
            nv.kern_fwd(0, X, None, ell, s2, noise=noise, lower=True, out=buf, ldk=ld)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            state["dinv"], info = nv.potrf_(buf, ld)
            e1.record()
            torch.cuda.synchronize()
            assert int(info.item()) == 0
            state.setdefault("potrf", []).append(e0.elapsed_time(e1))
            e0.record()
            nv.potri_(buf, ld, state["dinv"])
            e1.record()
            torch.cuda.synchronize()
            state.setdefault("potri", []).append(e0.elapsed_time(e1))

        potrf()                                  # warm-up (workspaces, tensor maps)
        state.clear()
        for _ in range(reps):
            potrf()
        med = {k: sorted(v)[len(v) // 2] for k, v in state.items() if k in ("potrf", "potri")}
        r = {"potrf_ms": med["potrf"], "potri_ms": med["potri"], "potrf_all_ms": state["potrf"],
             "potri_all_ms": state["potri"], "device_used_bytes": device_used_bytes(),
             "potrf_fp64_equiv_tflops": n ** 3 / 3.0 / med["potrf"] * 1e-9,
             "potri_fp64_equiv_tflops": 2.0 * n ** 3 / 3.0 / med["potri"] * 1e-9}
        if eng != "dmma":
            s_inv = INVERSE_SLICES if eng == "native" else slices
            r["potri_slices"] = s_inv
            r["potrf_int8_tops"] = r["potrf_fp64_equiv_tflops"] * slices * (slices + 1) / 2
            r["potri_int8_tops"] = r["potri_fp64_equiv_tflops"] * s_inv * (s_inv + 1) / 2
        res[eng] = r
        use("dmma", slices)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--slices", type=int, default=8)
    ap.add_argument("--sizes", default="16384,32768")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    prev = nv.i8mma_config(-1)
    out = {"card": card(), "slices": a.slices, "reps": a.reps}
    try:
        out["syrk_m30720_k2048"] = syrk_case(30720, 2048, a.slices, a.reps)
        print(json.dumps({"syrk_m30720_k2048": out["syrk_m30720_k2048"]}), flush=True)
        for n in [int(s) for s in a.sizes.split(",") if s]:
            out["potrf_potri_n%d" % n] = factor_case(n, a.slices, a.reps)
            print(json.dumps({"potrf_potri_n%d" % n: out["potrf_potri_n%d" % n]}), flush=True)
            torch.cuda.empty_cache()
    finally:
        nv.ozaki_config(0)
        nv.i8mma_config(prev)
    print(json.dumps(out["card"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
