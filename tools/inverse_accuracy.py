"""The error table of DESIGN.md section 8 for the engine the environment selects (GPB_OZAKI / GPB_I8MMA as set by the
caller): how far the consumers of the blocked inverse land from their references, each next to the tolerance the suite
holds it to.

- n16384_grad: GPR Rbf-ARD loss+grad at N = 16384 against the unmodified reference's gradients (tests/golden), tol 1e-7;
- n32768_residual: || Ky^-1 (Ky v) - v || / || v || (max norms) with Ky^-1 from gpb_potri_lower at N = 32768, tol 1e-8;
- n8192_posterior_var: GPR.posterior()'s variance (through Ky^-1) against predict_f's (triangular solves) at N = 8192
  on the UCB test's model and candidates, relative to the largest variance; and the UCB ascent's path, tol 1e-9.

    python tools/inverse_accuracy.py --out FILE                  # the default engine (factor 8 slices, inverse 9)
    GPB_OZAKI=9 python tools/inverse_accuracy.py --out FILE      # the library engine, factor and inverse at 9
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


def grad_n16384():
    from conftest import Cases
    from oracle import gp_oracle as O
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import GPR
    c, nm = Cases("large_cases.npz"), "gpr_n16384"
    X, Y, _ = O.synth_regression(16384, 8)
    model = GPR(X.numpy(), Y.numpy(), kernels.Rbf(8, ARD=True), likelihood=likelihoods.Gaussian(variance=0.01))
    loss = model.loss()
    loss.backward()
    ref_loss = float(np.asarray(c.get(nm, "loss")).ravel()[0])
    e = {"loss": abs(loss.item() - ref_loss) / abs(ref_loss),
         "g_variance": rel_err(model.kernel.variance.grad.cpu().numpy(), c.get(nm, "g_variance")),
         "g_length_scales": rel_err(model.kernel.length_scales.grad.cpu().numpy(), c.get(nm, "g_length_scales")),
         "g_noise": rel_err(model.likelihood.variance.grad.cpu().numpy(), c.get(nm, "g_noise"))}
    return {"errors": e, "worst_grad": max(e["g_variance"], e["g_length_scales"], e["g_noise"]), "tol": 1e-7}


def residual_n32768():
    from oracle import gp_oracle as O
    from gptorch_b200 import _native as nv
    n, d = 32768, 8
    X, _, _ = O.synth_regression(n, d)
    Xc = X.cuda()
    ell = torch.ones(d, dtype=torch.float64, device="cuda")
    s2 = torch.ones(1, dtype=torch.float64, device="cuda")
    noise = torch.full((1,), 0.01, dtype=torch.float64, device="cuda")
    buf, ld = nv._aligned_empty(n, n, Xc.device)
    nv.kern_fwd(0, Xc, None, ell, s2, noise=noise, out=buf, ldk=ld)
    v = torch.randn(n, 1, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    Kv = buf[:, :n] @ v
    dinv, info = nv.potrf_(buf, ld)
    assert int(info.item()) == 0
    kd = nv.potri_(buf, ld, dinv)
    Kinv = nv.potri_assemble(buf, ld, kd)
    r = rel_err((Kinv @ Kv).cpu().numpy(), v.cpu().numpy())
    del buf, Kinv
    torch.cuda.empty_cache()
    return {"residual": r, "tol": 1e-8}


def posterior_n8192():
    import test_gpu_posterior as T
    n, d, ns, beta = 8192, 8, 16, 2.0
    X, Y = T._data(n, d, 1)
    ell = 0.4 * np.sqrt(d) + 0.05 * np.arange(d)
    model = T._model(T._kern("Rbf", d, ell, 1.3, True), X, Y, 0.05)
    post = model.posterior()
    start = T._test_points(X, ns, seed=3).cuda()
    with torch.no_grad():
        _, v_post = post.predict_f(start)
        _, v_f = model.predict_f(start)
    var_rel = rel_err(v_post.cpu().numpy(), v_f.cpu().numpy())

    def ascend(source):
        x = start.clone().requires_grad_(True)
        opt = torch.optim.Adam([x], lr=0.05)
        for _ in range(5):
            opt.zero_grad()
            mean, var = source.predict_f(x)
            (-(mean + beta * var.clamp_min(1e-30).sqrt())).sum().backward()
            opt.step()
        return x.detach().cpu()

    path = rel_err(ascend(post).numpy(), ascend(model).numpy())
    return {"variance_vs_predict_f": var_rel, "ucb_path": path, "tol": 1e-9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"env": {k: os.environ.get(k) for k in ("GPB_OZAKI", "GPB_I8MMA")}, "gpu": torch.cuda.get_device_name(0)}
    for name, fn in (("n8192_posterior", posterior_n8192), ("n16384_grad", grad_n16384),
                     ("n32768_residual", residual_n32768)):
        res[name] = fn()
        torch.cuda.empty_cache()
        print(name, json.dumps(res[name]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
