"""cfg1 / cfg2 / cfg4 timings on the GPU, and the real reference on the host cores.
usage: python scripts/gpu_small_configs.py [out.json]"""
import contextlib, io, json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from oracle import ref, ref_inputs
from gglasso_b200 import ADMM_MGL, ADMM_SGL
from gglasso_b200.parallel import grid_search_device

out = {}


def quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def wall(fn, reps=3):
    best = 1e9
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter(); r = fn(); torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best, r


ADMM_MGL_ref, ADMM_SGL_ref, _ = ref.fresh_solvers()
S1 = ref_inputs.load("cfg1")
S2g, S2f = ref_inputs.load("cfg2_ggl"), ref_inputs.load("cfg2_fgl")
Om1 = np.eye(100); Om2 = np.repeat(np.eye(100)[None], 5, 0)
cases = {
    "cfg1_sgl": (lambda: quiet(ADMM_SGL, S1, 0.05, Om1, tol=1e-7, rtol=1e-7), lambda: quiet(ADMM_SGL_ref, S1, 0.05, Om1, tol=1e-7, rtol=1e-7)),
    "cfg2_ggl": (lambda: quiet(ADMM_MGL, S2g, 0.05, 0.01, "GGL", Om2, tol=1e-7, rtol=1e-7), lambda: quiet(ADMM_MGL_ref, S2g, 0.05, 0.01, "GGL", Om2, tol=1e-7, rtol=1e-7)),
    "cfg2_ggl_latent": (lambda: quiet(ADMM_MGL, S2g, 0.05, 0.01, "GGL", Om2, tol=1e-7, rtol=1e-7, latent=True, mu1=0.1), lambda: quiet(ADMM_MGL_ref, S2g, 0.05, 0.01, "GGL", Om2, tol=1e-7, rtol=1e-7, latent=True, mu1=0.1)),
    "cfg2_fgl": (lambda: quiet(ADMM_MGL, S2f, 0.05, 0.01, "FGL", Om2, tol=1e-7, rtol=1e-7), lambda: quiet(ADMM_MGL_ref, S2f, 0.05, 0.01, "FGL", Om2, tol=1e-7, rtol=1e-7)),
}
for name, (gpu, cpu) in cases.items():
    rec = {}
    gpu()
    rec["gpu_s"], (sol, info) = wall(gpu)
    cpu()
    rec["cpu_reference_s"], (rsol, rinfo) = wall(cpu, reps=2)
    rec["theta_rel_err"] = float(np.linalg.norm(sol["Theta"] - rsol["Theta"]) / np.linalg.norm(rsol["Theta"]))
    rec["speedup"] = rec["cpu_reference_s"] / rec["gpu_s"]
    print(name, rec, flush=True)
    out[name] = rec

S4 = ref_inputs.load("cfg4"); N4 = np.full(10, 1000)
l1, l2 = np.logspace(0, -3, 10), np.logspace(-1, -4, 10)
for ns in (5, 10, 3, 1):
    grid_search_device(S4, N4, "GGL", l1[4:5], l2[:2], gamma=0.1, tol=1e-5, rtol=1e-5)
    t, (scores, iters, ix, best) = wall(lambda: grid_search_device(S4, N4, "GGL", l1, l2, gamma=0.1, tol=1e-7, rtol=1e-7, n_streams=ns), reps=1)
    rec = {"n_streams": ns, "seconds": t, "iterations": int(iters.sum()), "best": [int(i) for i in ix]}
    print("cfg4_grid", rec, flush=True)
    out[f"cfg4_grid_streams{ns}"] = rec
json.dump(out, open(sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/small_configs.json", "w"), indent=1)
