"""ADMM_MGL_batch measurements -> profiles/r05_mgl_batch.json (or the path given as argv[1]).

For each shape, three arms solve the same B problems to tol = rtol = 1e-7 (Omega_0 = I, cold start):
  batch       one ADMM_MGL_batch call;
  sequential  B ADMM_MGL calls, one after the other;
  threads5    the B ADMM_MGL calls dealt round-robin to 5 host threads, each on its own CUDA stream (what
              grid_search_device(n_streams=5) does with the columns of a grid).
Shapes:
  cfg2_ggl_bootB   GGL K=5 p=100, lambda1 = 0.05, lambda2 = 0.01, B in {1, 10, 100} parametric-bootstrap covariances
                   (N = 1000 draws from N(0, S_k + 1e-3 I), S = the reference-generated cfg2 input);
  cfg4_l1_path     GGL K=10 p=500, the ten lambda1 of the cfg4 grid (logspace(0, -3, 10)) at lambda2 = 0.1, the
                   reference-generated cfg4 input;
  cfg3_B2          FGL K=20 p=1000, (lambda1, lambda2) = (0.05, 0.01) and (0.1, 0.01), the reference-generated cfg3 input.
Every arm runs once untimed per shape first; the timed repetitions alternate the arms (REPS rounds).  Reported: wall
seconds per repetition, total problem-iterations, ms per problem-iteration, and whether every problem's outputs of the
batch are bitwise those of its ADMM_MGL call (and otherwise the largest relative difference).
"""
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gglasso_b200 import ADMM_MGL, ADMM_MGL_batch  # noqa: E402
from oracle import ref_inputs  # noqa: E402

TOL = 1e-7
REPS = 3
STREAMS = 5


def bootstrap(S, B, N=1000, seed=0):
    rng = np.random.default_rng(seed)
    K, p, _ = S.shape
    out = np.empty((B, K, p, p))
    for k in range(K):
        C = np.linalg.cholesky(S[k] + 1e-3 * np.eye(p))
        for b in range(B):
            Z = rng.standard_normal((N, p)) @ C.T
            out[b, k] = Z.T @ Z / N
    return out


def shapes():
    s2 = ref_inputs.load("cfg2_ggl")
    boot = bootstrap(s2, 100)
    for B in (1, 10, 100):
        yield f"cfg2_ggl_boot{B}", boot[:B], "GGL", np.full(B, 0.05), np.full(B, 0.01)
    yield "cfg4_l1_path", ref_inputs.load("cfg4"), "GGL", np.logspace(0, -3, 10), np.full(10, 0.1)
    yield "cfg3_B2", ref_inputs.load("cfg3"), "FGL", np.array([0.05, 0.1]), np.array([0.01, 0.01])


def one(S, b):
    return S[b] if S.ndim == 4 else S


def arm_batch(S, reg, l1, l2, eye, max_iter):
    return ADMM_MGL_batch(S, l1, l2, reg, eye, tol=TOL, rtol=TOL, max_iter=max_iter)


def _single(S, reg, l1, l2, eye, b, max_iter):
    return ADMM_MGL(one(S, b), float(l1[b]), float(l2[b]), reg, eye, tol=TOL, rtol=TOL, max_iter=max_iter)


def arm_sequential(S, reg, l1, l2, eye, max_iter):
    return [_single(S, reg, l1, l2, eye, b, max_iter) for b in range(len(l1))]


def arm_threads(S, reg, l1, l2, eye, max_iter):
    B = len(l1)
    out = [None] * B
    errs = []

    def work(bs):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for b in bs:
                    out[b] = _single(S, reg, l1, l2, eye, b, max_iter)
                torch.cuda.current_stream().synchronize()
        except Exception as ex:
            errs.append(ex)

    ts = [threading.Thread(target=work, args=(list(range(w, B, STREAMS)),)) for w in range(min(STREAMS, B))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    if errs:
        raise errs[0]
    return out


def run_arm(fn, *args):
    """(iteration counts, results): ADMM_MGL prints its iteration count; the threads' lines come in any order, so
    the counts are returned sorted"""
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        res = fn(*args)
    if fn is arm_batch:
        return [len(i["residual"]) for _, i in res], res
    n = [int(t.split()[0]) for t in buf.getvalue().split("ADMM terminated after ")[1:]]
    return (sorted(n) if fn is arm_threads else n), res


ARMS = {"batch": arm_batch, "sequential": arm_sequential, "threads5": arm_threads}


def main(path):
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    rec = {"gpu": gpu, "torch": torch.__version__, "tol": TOL, "rtol": TOL, "reps": REPS, "streams": STREAMS,
           "what": __doc__.strip(), "shapes": {}}
    for name, S, reg, l1, l2 in shapes():
        K, p = S.shape[-3], S.shape[-1]
        eye = np.repeat(np.eye(p)[None], K, 0)
        for fn in ARMS.values():                        # warm-up of every arm at this shape
            run_arm(fn, S, reg, l1, l2, eye, 5)
        torch.cuda.synchronize()
        times = {a: [] for a in ARMS}
        iters, outs = {}, {}
        for _ in range(REPS):
            for a, fn in ARMS.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                n, res = run_arm(fn, S, reg, l1, l2, eye, 1000)
                torch.cuda.synchronize()
                times[a].append(time.perf_counter() - t0)
                iters[a], outs[a] = n, res
        bitwise, worst = True, 0.0
        for (sb, ib), (ss, is_) in zip(outs["batch"], outs["sequential"]):
            assert ib["status"] == is_["status"]
            for k in ("Omega", "Theta", "X"):
                bitwise &= bool(np.array_equal(sb[k], ss[k]))
                worst = max(worst, float(np.linalg.norm(sb[k] - ss[k]) / max(np.linalg.norm(ss[k]), 1e-300)))
        r = {"K": K, "p": p, "reg": reg, "B": len(l1), "lambda1": l1.tolist(), "lambda2": l2.tolist(),
             "seconds": times, "iterations": iters, "bitwise_equal_to_ADMM_MGL": bitwise, "max_rel_diff": worst,
             "same_iterations": (iters["batch"] == iters["sequential"]
                                 and sorted(iters["batch"]) == iters["threads5"])}
        tot = sum(iters["batch"])
        r["problem_iterations"] = tot
        r["ms_per_problem_iteration"] = {a: 1e3 * min(t) / tot for a, t in times.items()}
        r["best_seconds"] = {a: min(t) for a, t in times.items()}
        rec["shapes"][name] = r
        print(name, json.dumps({k: r[k] for k in ("best_seconds", "ms_per_problem_iteration", "problem_iterations",
                                                  "bitwise_equal_to_ADMM_MGL", "max_rel_diff")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r05_mgl_batch.json"))
