"""stage 1 as concurrent chains over groups of the batch: CUDA-event times of gg_eigh and of the tridiagonalisation
alone (gg_sytrd_profile(which=0)), the host time to enqueue one gg_eigh call (host clock, no synchronise) and the
eigenvalue error against LAPACK, at the batch shapes of the benchmark and around it.  GGLASSO_B200_LIB selects another
build of the library (A/B runs against the parent's build).
usage: python scripts/gpu_tr_groups.py [out.json]   (default: tr_groups.json in the current directory)"""
import json, os, subprocess, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gglasso_b200 import _lib
from gglasso_b200._engine import Eigh, to_dev, _p

SHAPES = ((20, 1000), (10, 1000), (3, 1000), (10, 500), (6, 384), (2, 2047), (1, 1384))
REPS = 8

lib = _lib.load()
dev = torch.device("cuda")
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
except Exception:
    gpu = torch.cuda.get_device_name()
out = {"gpu": gpu, "lib": _lib.LIB_PATH, "reps": REPS, "statistic": "median", "shapes": []}


def sym(rng, M, p):
    A = rng.standard_normal((M, p, p))
    return (A + A.transpose(0, 2, 1)) / 2


for M, p in SHAPES:
    rng = np.random.default_rng(p + M)
    A = sym(rng, M, p)
    e = Eigh(M, p, dev)
    st = torch.cuda.current_stream().cuda_stream
    A0 = to_dev(A, dev)
    W = A0.clone()
    D = e.eigh(W, stream=st)
    torch.cuda.synchronize()
    rec = {"M": M, "p": p,
           "eig_err": float(np.abs(np.sort(D.cpu().numpy(), 1) - np.linalg.eigvalsh(A)).max())}
    calls = (("eigh", lambda W: e.eigh(W, stream=st)),
             ("sytrd", lambda W: _lib.check(lib.gg_sytrd_profile(_p(W), _p(e.D), M, p, _p(e.ws), e.ws_bytes, 0, st),
                                            "gg_sytrd_profile")))
    for name, fn in calls:
        dts, hts = [], []
        for r in range(REPS + 1):
            W = A0.clone()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            h0 = time.perf_counter()
            fn(W)
            h1 = time.perf_counter()
            b.record()
            torch.cuda.synchronize()
            if r:
                dts.append(a.elapsed_time(b))
                hts.append((h1 - h0) * 1e3)
        rec[f"{name}_ms"] = float(np.median(dts))
        rec[f"{name}_ms_spread"] = [float(min(dts)), float(max(dts))]
        rec[f"{name}_host_enqueue_ms"] = float(np.median(hts))
    print(json.dumps(rec), flush=True)
    out["shapes"].append(rec)
    del e, W, A0
    torch.cuda.empty_cache()
json.dump(out, open(sys.argv[1] if len(sys.argv) > 1 else "tr_groups.json", "w"), indent=1)
