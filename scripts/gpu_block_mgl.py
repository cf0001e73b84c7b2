"""block_MGL measurements -> profiles/r07_block_mgl.json (or the path given as argv[1]).

Inputs: gglasso_b200.datagen.synthetic_mgl, K = 5, p = 1000 and p = 5000 (blocks of 100 nodes), GGL on kind='group'
and FGL on kind='fused' covariances, lambda2 = lambda1 / 5.  For each input two lambda1 are taken from a fixed
candidate list by the screen itself: 'small' = the smallest candidate whose largest component has <= 160 nodes (many
small components, all in ragged batches), 'large' = the largest candidate with a component above 160 nodes (a few
large components, one at a time on the large-p path).

Recorded per case:
  screen_ms            gg_mgl_screen alone, CUDA events (S already on the device), best of 5
  components_ms        host component search from the bitmask (scipy), best of 5
  batches_s, large_s   wall seconds block_MGL spends in its ragged batches and in its large components (one timed call)
  block_mgl_s          block_MGL wall seconds, ADMM_MGL_s the full problem's, tol = rtol = 1e-7, Omega_0 = I; one
                       untimed call of each first, then best of REPS alternating repetitions (a single timed repetition
                       when one ADMM_MGL call takes longer than SLOW_S)
  sizes                component-size histogram (bucket upper edge -> count; sizes above 160 listed)
  theta_rel_diff       |Theta_block - Theta_full|_F / |Theta_full|_F, pattern_equal: identical nonzero pattern
The GPU name, power limit and maximum SM clock are read with nvidia-smi in the same run.
"""
import contextlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gglasso_b200 import ADMM_MGL, block_MGL, _lib  # noqa: E402
from gglasso_b200._engine import _p, to_dev  # noqa: E402
from gglasso_b200.datagen import synthetic_mgl  # noqa: E402
from gglasso_b200.solver import admm_solver  # noqa: E402

TOL = 1e-7
REPS = 3
SLOW_S = 30.0
K = 5
CANDIDATES = [0.2, 0.15, 0.1, 0.07, 0.05, 0.035, 0.025, 0.018, 0.012]
EDGES = [1, 2, 4, 8, 16, 32, 64, 96, 128, 160]


def quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def screen_ms(Sd, l1, l2, reg):
    lib = _lib.load()
    p = Sd.shape[1]
    adj = torch.empty((p, (p + 31) // 32), dtype=torch.int32, device=Sd.device)
    st = torch.cuda.current_stream()
    best = float("inf")
    for _ in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        _lib.check(lib.gg_mgl_screen(_p(Sd), None, l1, l2, 0 if reg == "GGL" else 1, K, p, _p(adj), st.cuda_stream),
                   "gg_mgl_screen")
        b.record(st)
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    words = adj.cpu().numpy().view(np.uint32)
    t = []
    for _ in range(5):
        t0 = time.perf_counter()
        numC, allC = admm_solver._components_from_bitmask(words, p)
        t.append(time.perf_counter() - t0)
    return best, 1e3 * min(t), allC


def histogram(allC):
    sizes = np.array([len(C) for C in allC])
    h = {str(e): int(((sizes <= e) & (sizes > lo)).sum()) for lo, e in zip([0] + EDGES[:-1], EDGES)}
    return {"buckets": h, "above_160": sorted(int(s) for s in sizes[sizes > 160])}


class Timed:
    """accumulates the wall time of calls to one module function while installed"""
    def __init__(self, name):
        self.name, self.orig, self.total = name, getattr(admm_solver, name), 0.0

    def __enter__(self):
        def wrap(*a, **kw):
            t0 = time.perf_counter()
            try:
                return self.orig(*a, **kw)
            finally:
                self.total += time.perf_counter() - t0
        setattr(admm_solver, self.name, wrap)
        return self

    def __exit__(self, *exc):
        setattr(admm_solver, self.name, self.orig)


def case(S, reg, l1, allC, s_ms, c_ms):
    l2 = l1 / 5
    p = S.shape[1]
    eye = np.repeat(np.eye(p)[None], K, 0)
    kw = dict(tol=TOL, rtol=TOL)
    t0 = time.perf_counter()
    full, finfo = quiet(ADMM_MGL, S, l1, l2, reg, eye, **kw)                  # untimed warm-up of each arm
    t_first_full = time.perf_counter() - t0
    with Timed("_solve_mgl_batch") as tb, Timed("_solve_mgl_large") as tl:
        blk, binfo = quiet(block_MGL, S, l1, l2, reg, eye, **kw)
    reps = REPS if t_first_full < SLOW_S else 1
    tb_, tf_ = [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        blk, binfo = quiet(block_MGL, S, l1, l2, reg, eye, **kw)
        tb_.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        full, finfo = quiet(ADMM_MGL, S, l1, l2, reg, eye, **kw)
        tf_.append(time.perf_counter() - t0)
    n_full = np.linalg.norm(full["Theta"])
    return {
        "lambda1": l1, "lambda2": l2, "n_components": len(allC), "sizes": histogram(allC),
        "screen_ms": s_ms, "components_ms": c_ms, "batches_s": tb.total, "large_s": tl.total,
        "block_mgl_s": min(tb_), "ADMM_MGL_s": min(tf_), "reps": reps,
        "block_mgl_s_all": tb_, "ADMM_MGL_s_all": tf_,
        "speedup": min(tf_) / min(tb_),
        "status_block": binfo["status"], "status_full": finfo["status"],
        "max_component_iters": int(np.max(binfo["component_iters"])),
        "theta_rel_diff": float(np.linalg.norm(blk["Theta"] - full["Theta"]) / n_full),
        "pattern_equal": bool(np.array_equal(blk["Theta"] != 0, full["Theta"] != 0)),
    }


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_block_mgl.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    res = {"gpu": gpu, "torch": torch.__version__, "tol": TOL, "rtol": TOL, "K": K, "candidates": CANDIDATES,
           "what": __doc__, "cases": []}
    for p in (1000, 5000):
        for reg, kind in (("GGL", "group"), ("FGL", "fused")):
            S = synthetic_mgl(K, p, seed=0, kind=kind, n_blocks=p // 100)
            Sd = to_dev(S, torch.device("cuda"))
            scan = {}
            for l1 in CANDIDATES:
                scan[l1] = screen_ms(Sd, l1, l1 / 5, reg)
            maxsize = {l1: max(len(C) for C in v[2]) for l1, v in scan.items()}
            small = min((l1 for l1 in CANDIDATES if maxsize[l1] <= 160), default=None)
            large = max((l1 for l1 in CANDIDATES if maxsize[l1] > 160), default=None)
            del Sd
            for label, l1 in (("small", small), ("large", large)):
                if l1 is None:
                    continue
                s_ms, c_ms, allC = scan[l1]
                r = case(S, reg, l1, allC, s_ms, c_ms)
                r.update(p=p, reg=reg, kind=kind, regime=label)
                res["cases"].append(r)
                print(json.dumps({k: r[k] for k in ("p", "reg", "regime", "lambda1", "n_components", "screen_ms",
                                                     "components_ms", "batches_s", "large_s", "block_mgl_s",
                                                     "ADMM_MGL_s", "speedup", "theta_rel_diff", "pattern_equal")}),
                      flush=True)
            res["scan_" + f"{reg}_p{p}"] = {str(l1): {"max_component": maxsize[l1], "n_components": len(scan[l1][2]),
                                                     "screen_ms": scan[l1][0]} for l1 in CANDIDATES}
            with open(out_path, "w") as f:
                json.dump(res, f, indent=1)
    print(gpu)


if __name__ == "__main__":
    main()
