"""stability_selection measurements -> profiles/r06_stars.json (or the path given as argv[1]).

For each shape, L = 10 values of lambda1 (logspace(-0.3, -1.5, 10)) and B = 20 subsamples of the default size
(floor(10 sqrt(n)) rows per class), scale=True, tol = rtol = 1e-7, Omega_0 = I:
  a_device      stability_selection(..., refit=False): samples, covariances, solves and edge counts on the device;
  b_host        the host composition: numpy subsample covariances (same indices), then ADMM_MGL_batch on the B*L
                problems (MGL) or B*L ADMM_SGL calls (SGL), then counting and instabilities in numpy;
  c_sequential  (MGL) B*L sequential ADMM_MGL calls on the same covariances, solves only.  For SGL the solves of b_host
                are already B*L sequential ADMM_SGL calls; their time is reported as c_sequential_within_b.
Shapes: SGL p=100 n=200 and p=500 n=1000; MGL GGL and FGL K=5 p=100 n_k=200 at lambda2 = 0.01; MGL GGL K=10 p=500
n_k=1000 at lambda2 = 0.01.  Samples: Gaussian draws from datagen.instance_precisions (seeded).
Every arm runs once untimed per shape first; the timed repetitions alternate the arms (REPS rounds), best of REPS is
reported.  a_device is checked against b_host: best index, mean edges (= summed counts / B) and instability per
lambda1, and the edge counts at the selected lambda1.

gg_subsample_cov alone: the B covariances of each shape, timed with CUDA events over 20 launches after a warm-up (the
samples fit in L2).  FLOP counts: the full product 2 b p^2 K per subsample, and the upper tiles the kernel computes,
2 b K p^2 * (nt + 1) / (2 nt) with nt = ceil(p/64) tiles per side; rates against the 37.0 TFLOP/s DMMA issue peak of
profiles/r02_dmma_peak.jsonl.
"""
import contextlib
import io
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gglasso_b200 import ADMM_MGL, ADMM_MGL_batch, ADMM_SGL, datagen, stability_selection  # noqa: E402
from gglasso_b200 import stability as stars  # noqa: E402
from gglasso_b200 import _lib  # noqa: E402

TOL = 1e-7
REPS = 3
L_PATH = np.logspace(-0.3, -1.5, 10)
B = 20
DMMA_PEAK = 37.0e12


def samples(K, p, n, seed, kind="group"):
    Th = datagen.instance_precisions(K, p, n_blocks=10, seed=seed, kind=kind)
    rng = np.random.default_rng(seed + 7)
    out = []
    for k in range(K):
        Lc = np.linalg.cholesky(Th[k])
        out.append(np.linalg.solve(Lc.T, rng.standard_normal((p, n))).T.copy())
    return out


def shapes():
    yield "sgl_p100_n200", samples(1, 100, 200, 1)[0], None, None
    yield "sgl_p500_n1000", samples(1, 500, 1000, 2)[0], None, None
    yield "mgl_ggl_K5_p100_n200", samples(5, 100, 200, 3), "GGL", 0.01
    yield "mgl_fgl_K5_p100_n200", samples(5, 100, 200, 4, kind="fused"), "FGL", 0.01
    yield "mgl_ggl_K10_p500_n1000", samples(10, 500, 1000, 5), "GGL", 0.01


def counts_np(Th):
    p = Th.shape[-1]
    iu = np.triu_indices(p, 1)
    C = np.zeros(Th.shape[1:], dtype=np.int64)
    C[..., iu[0], iu[1]] = (Th[..., iu[0], iu[1]] != 0).sum(0)
    return C


def arm_a(data, reg, l2, max_iter=1000):
    return stability_selection(data, L_PATH, lambda2=l2, reg=reg, n_subsamples=B, refit=False, tol=TOL, rtol=TOL,
                               max_iter=max_iter)


def host_covs(data, reg):
    classes = [data] if reg is None else data
    b = [stars.default_subsample_size(x.shape[0]) for x in classes]
    idx = stars.draw_indices([x.shape[0] for x in classes], b, B, 0)
    return np.stack([np.stack([stars.sample_covariance(x[idx[k][s]], True) for k, x in enumerate(classes)])
                     for s in range(B)])                     # (B, K, p, p)


def solve_host(S, reg, l2, lam, max_iter):
    """(B, L, K, p, p) Theta of every problem, and the seconds spent in the solver calls"""
    Bn, K, p, _ = S.shape
    L = len(lam)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        if reg is None:
            Th = np.stack([[ADMM_SGL(S[s, 0], lam[l], np.eye(p), tol=TOL, rtol=TOL, max_iter=max_iter)[0]["Theta"]
                            for l in range(L)] for s in range(Bn)])[:, :, None]
        else:
            out = ADMM_MGL_batch(np.repeat(S, L, axis=0), np.tile(lam, Bn), l2, reg, np.repeat(np.eye(p)[None], K, 0),
                                 tol=TOL, rtol=TOL, max_iter=max_iter)
            Th = np.stack([sol["Theta"] for sol, _ in out]).reshape(Bn, L, K, p, p)
    return Th, time.perf_counter() - t0


def arm_b(data, reg, l2, max_iter=1000):
    lam = np.sort(L_PATH)[::-1]
    S = host_covs(data, reg)
    Th, t_solve = solve_host(S, reg, l2, lam, max_iter)
    C = counts_np(Th)
    p = C.shape[-1]
    iu = np.triu_indices(p, 1)
    th = C[..., iu[0], iu[1]] / B
    D_k = (2 * th * (1 - th)).sum(-1) / (p * (p - 1) / 2)
    D = D_k.mean(1)
    _, best = stars.select(D, 0.05)
    return dict(C=C, D=D, E=C[..., iu[0], iu[1]].sum(-1) / B, best=best, t_solve=t_solve, S=S)


def arm_c(data, reg, l2, S, max_iter=1000):
    lam = np.sort(L_PATH)[::-1]
    K, p = S.shape[1], S.shape[-1]
    eye = np.repeat(np.eye(p)[None], K, 0)
    with contextlib.redirect_stdout(io.StringIO()):
        for s in range(B):
            for l in lam:
                ADMM_MGL(S[s], l, l2, reg, eye, tol=TOL, rtol=TOL, max_iter=max_iter)


def time_cov(data, reg):
    classes = [data] if reg is None else data
    K, p = len(classes), classes[0].shape[1]
    b = [stars.default_subsample_size(x.shape[0]) for x in classes]
    idx = stars.draw_indices([x.shape[0] for x in classes], b, B, 0)
    res = stars._Resident(classes, idx, torch.device("cuda"))
    lib = _lib.load()
    S = torch.empty((B * K, p, p), dtype=torch.float64, device="cuda")
    mean = torch.empty((B * K, p), dtype=torch.float64, device="cuda")
    zc = torch.empty(B * K, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    P = stars._p
    out = {}
    for scale in (0, 1):
        def go():
            _lib.check(lib.gg_subsample_cov(P(res.X), P(res.rowoff), P(res.idx), P(res.boff), B, K, p, scale,
                                            P(mean), P(S), P(zc), st), "gg_subsample_cov")
        for _ in range(3):
            go()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 20
        e0.record()
        for _ in range(n):
            go()
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) / 1e3 / n
        nt = (p + 63) // 64
        full = float(sum(2.0 * bk * p * p for bk in b) * B)
        upper = full * (nt + 1) / (2 * nt)
        out["scaled" if scale else "unscaled"] = {
            "seconds": sec, "flops_full_product": full, "flops_upper_tiles": upper,
            "tflops_full_equivalent": full / sec / 1e12, "tflops_upper_tiles": upper / sec / 1e12,
            "share_of_dmma_peak_upper_tiles": upper / sec / DMMA_PEAK}
    return out


def main(path):
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    rec = {"gpu": gpu, "torch": torch.__version__, "tol": TOL, "rtol": TOL, "reps": REPS, "B": B,
           "lambda1": L_PATH.tolist(), "what": __doc__.strip(), "shapes": {}}
    print("gpu:", gpu, flush=True)
    for name, data, reg, l2 in shapes():
        is_sgl = reg is None
        arms = ["a_device", "b_host"] + ([] if is_sgl else ["c_sequential"])
        # warm-up of every arm at this shape (max_iter = 5: the max-iterations warnings are expected)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            arm_a(data, reg, l2, 5)
        wb = arm_b(data, reg, l2, 5)
        if not is_sgl:
            arm_c(data, reg, l2, wb["S"], 5)
        torch.cuda.synchronize()
        times = {a: [] for a in arms}
        if is_sgl:
            times["c_sequential_within_b"] = []
        for _ in range(REPS):
            for a in arms:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if a == "a_device":
                    ra = arm_a(data, reg, l2)
                elif a == "b_host":
                    rb = arm_b(data, reg, l2)
                else:
                    arm_c(data, reg, l2, rb["S"])
                torch.cuda.synchronize()
                times[a].append(time.perf_counter() - t0)
            if is_sgl:
                times["c_sequential_within_b"].append(rb["t_solve"])
        best = ra["best_index"]
        Cb = rb["C"][best]
        ef = ra["edge_frequency"][None] if is_sgl else ra["edge_frequency"]
        match = {"best_index": best == rb["best"],
                 "edge_counts_at_best": bool(np.array_equal(ef * B, (Cb + Cb.transpose(0, 2, 1)).astype(float))),
                 "mean_edges": bool(np.array_equal(ra["mean_edges"], rb["E"])),
                 "instability_max_rel_diff": float(np.max(np.abs(ra["instability"] - rb["D"])
                                                          / np.maximum(np.abs(rb["D"]), 1e-300)))}
        r = {"K": 1 if is_sgl else len(data), "p": int(ef.shape[-1]), "reg": reg or "SGL", "lambda2": l2,
             "seconds": times, "best_seconds": {a: min(t) for a, t in times.items()},
             "a_matches_b": match, "best_index": best, "instability": ra["instability"].tolist(),
             "mean_edges": ra["mean_edges"].mean(1).tolist(), "n_not_optimal": ra["n_not_optimal"].tolist(),
             "subsample_cov": time_cov(data, reg)}
        rec["shapes"][name] = r
        print(name, json.dumps({k: r[k] for k in ("best_seconds", "a_matches_b", "best_index")}),
              json.dumps(r["subsample_cov"]["scaled"]), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:                     # after every shape: a partial run keeps what it measured
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r06_stars.json"))
