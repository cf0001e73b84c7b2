"""Kernel-level tests of the ADMM loop's entry points that otherwise only whole solves check: each kernel is called
through the C ABI and compared with a host reference (oracle/kernel_refs.py, mpmath for eigenvalues, exact sums for
reductions), with sentinel regions around every output, problems marked done left untouched, and every case run
twice to show that the result is deterministic.

Tolerances: elementwise results bitwise; reductions against math.fsum within 1e-13 of the sum of absolute terms;
max-reductions bitwise; eigenpairs within C_EIG * sqrt(p) eps |A| (eigenvalues) and C_EIG * p eps |A| (residual,
orthogonality), |A| = max(|A|_2, |sigma|) with sigma the Gershgorin shift of the Jacobi solver (it only differs from
|A|_2 for multiples of the identity).  Setting GG_UNIT_REPORT=<path> writes the largest measured error ratios there."""
import ctypes
import json
import math
import os
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import kernel_refs as kr

pytestmark = pytest.mark.gpu

GUARD = 4096          # elements of sentinel before and after every output buffer
FILL = -7.25          # sentinel value
EPS = np.finfo(np.float64).eps
C_EIG = 8.0           # eigenpair tolerance constant (largest ratio measured on a B200: see DESIGN.md)
RTOL_SUM = 1e-13

_WORST = {}


def _note(key, value):
    _WORST[key] = max(_WORST.get(key, 0.0), float(value))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("GG_UNIT_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(_WORST, f, indent=1, sort_keys=True)


# ---- plumbing ----------------------------------------------------------------------------------------------------
def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _lib():
    from gglasso_b200 import _lib
    return _lib, _lib.load(), torch.cuda.current_stream().cuda_stream


def _dev(a, dtype=torch.float64):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dtype)


def _guarded(n, init=None, dtype=torch.float64):
    buf = torch.full((n + 2 * GUARD,), FILL, dtype=dtype, device="cuda")
    if init is not None:
        buf[GUARD:GUARD + n].copy_(torch.as_tensor(np.ascontiguousarray(init)).reshape(-1))
    return buf


def _inner(buf):
    return buf[GUARD:-GUARD]


def _guards_intact(buf):
    return bool((buf[:GUARD] == FILL).all()) and bool((buf[-GUARD:] == FILL).all())


def _out(bufs, shapes):
    """host copies of the guarded buffers' contents after checking their sentinels"""
    res = {}
    for k, b in bufs.items():
        assert _guards_intact(b), f"{k}: write outside the output"
        res[k] = _inner(b).cpu().numpy().reshape(shapes[k])
    return res


def _twice(run):
    """run a case twice; the results must be bitwise identical"""
    a, b = run(), run()
    for k in a:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), f"{k} differs"
    return a


def _ctrl_np(rho, xs=None, done=()):
    from gglasso_b200._lib import CTRL_STRIDE, C_RHO, C_XSCALE, C_DONE
    rho = np.asarray(rho, dtype=np.float64)
    c = np.zeros((rho.size, CTRL_STRIDE))
    c[:, C_RHO] = rho
    c[:, C_XSCALE] = 1.0 if xs is None else xs
    c[list(done), C_DONE] = 1.0
    c[:, 11:] = np.arange(5) + 0.5           # unused slots: must survive every kernel
    return c


def _sym(rng, n, p, scale=1.0):
    A = rng.standard_normal((n, p, p)) * scale
    return A + A.transpose(0, 2, 1)


def _same(a, b):
    """bitwise equality of two float64 arrays (NaN matches NaN whatever its payload)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))).all())


def _check_sums(got, ref, key, abs_ref=None):
    """sum of the kernel's partials against an exact sum"""
    err = abs(kr.fsum(got) - ref) / max(abs_ref if abs_ref is not None else abs(ref), 1e-300)
    _note(key, err)
    assert err <= RTOL_SUM, (key, err)


def _ew_multipass(M, p):
    """True when a CTA of the elementwise kernels makes more than one pass of its grid-stride loop"""
    need = -(-p * p // (256 * 4))
    cap = max((1184 + M - 1) // M, 1)
    return need > cap


# ======================================================================================================================
# 1. eigensolver: warm-started shared-memory Jacobi, block Jacobi
# ======================================================================================================================
def _jacobi_sweeps_offset(M, p):
    """byte offset of the per-matrix sweep counts the shared-memory Jacobi leaves in its workspace (layout of
    gg_jacobi_ws_bytes: sigma, rowlo, rowhi, conv, rotcount, maxoff, flags, sweeps)"""
    al = lambda x: (x + 255) // 256 * 256  # noqa: E731
    return al(8 * M) + 2 * al(8 * M * p) + 2 * al(4 * M) + al(8 * M) + 256


def _run_eigh(A, warm=None, nb2=0, vectors=1, ctrl=None, mpp=1, quad_tol=1e-10):
    _l, lib, st = _lib()
    M, p, _ = A.shape
    n = A.size
    ws_bytes = int(lib.gg_eigh_workspace_bytes(M, p))
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    bufs = {"Vt": _guarded(n, A), "D": _guarded(M * p)}
    if warm is not None:
        bufs["warm"] = _guarded(n, warm)
    info = (ctypes.c_int * 4)(-99, -99, -99, -99)
    cdev = _dev(ctrl)
    rc = lib.gg_eigh(_p(_inner(bufs["Vt"])), _p(_inner(bufs["D"])), M, p, _p(cdev), mpp, _p(ws), ws_bytes, vectors,
                     nb2, 0.0, 0, quad_tol, info, _p(_inner(bufs["warm"])) if warm is not None else None, st)
    _l.check(rc, "gg_eigh")
    torch.cuda.synchronize()
    out = _out(bufs, {"Vt": A.shape, "D": (M, p), "warm": A.shape})
    out["info"] = np.array([info[0]])
    if p <= 160 and (nb2 == 1 or p <= lib.gg_jacobi_max()):
        off = _jacobi_sweeps_offset(M, p)
        out["sweeps"] = ws[off:off + 4 * M].cpu().numpy().view(np.int32).copy()
    if cdev is not None:
        assert _same(cdev.cpu().numpy(), ctrl)
    return out


def _gersh_shift(a):
    d = np.diag(a)
    rs = np.abs(a).sum(axis=1) - np.abs(d)
    lo, hi = (d - rs).min(), (d + rs).max()
    c, h = 0.5 * (lo + hi), 0.5 * (hi - lo)
    if not h > 0:
        h = max(abs(c), 1.0)
    return 2 * h - c


_MP_CACHE = {}


def _ref_eigs(a):
    """eigenvalues of the stored matrix: mpmath at 34 digits for p <= 48, LAPACK above"""
    p = a.shape[0]
    if p > 48:
        return np.linalg.eigvalsh(a)
    key = a.tobytes()
    if key not in _MP_CACHE:
        import mpmath
        with mpmath.workdps(34):
            ev = mpmath.eigsy(mpmath.matrix(a.tolist()), eigvals_only=True)
            _MP_CACHE[key] = np.sort(np.array([float(x) for x in ev]))
    return _MP_CACHE[key]


def _check_eigpairs(A, Vt, D, tag):
    M, p, _ = A.shape
    worst = 0.0
    for m in range(M):
        a, v, d = A[m], Vt[m], D[m]
        scale = max(np.linalg.norm(a, 2), abs(_gersh_shift(a)))
        if scale == 0:
            scale = 1.0
        e = np.abs(np.sort(d) - _ref_eigs(a)).max() / (math.sqrt(p) * EPS * scale)
        res = np.linalg.norm(a @ v.T - v.T * d, axis=0).max() / (p * EPS * scale)
        orth = np.abs(v @ v.T - np.eye(p)).max() / (p * EPS)
        _note("eig_" + tag, e)
        _note("res_" + tag, res)
        _note("orth_" + tag, orth)
        worst = max(worst, e, res, orth)
        assert e <= C_EIG and res <= C_EIG and orth <= C_EIG, (tag, m, e, res, orth)
    return worst


SPECTRA = ("zero", "minus5", "three", "clustered", "negdef", "rankdef", "tiny", "huge", "offset")


def _spectra_stack(p, seed):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((p, p)))

    def qdq(d):
        a = (Q * d) @ Q.T
        return (a + a.T) / 2
    E = _sym(rng, 1, p)[0] / 2
    B = rng.standard_normal((p, max(p // 3, 1)))
    out = {"zero": np.zeros((p, p)), "minus5": -5 * np.eye(p), "three": 3 * np.eye(p),
           "clustered": qdq(1.0 + 1e-9 * rng.random(p)), "negdef": qdq(-rng.uniform(0.5, 4.0, p)),
           "rankdef": B @ B.T if p > 2 else np.zeros((p, p)), "tiny": 1e-8 * E, "huge": 1e8 * E,
           "offset": 1e6 * np.eye(p) + E}
    return np.stack([out[k] for k in SPECTRA])


def _warm_starts(A, seed):
    """name -> (M,p,p) warm start (rows orthonormal)"""
    rng = np.random.default_rng(seed + 1)
    M, p, _ = A.shape
    exact = np.linalg.eigh(A)[1].transpose(0, 2, 1).copy()
    pert = np.linalg.eigh(A + 1e-6 * np.linalg.norm(A, axis=(1, 2), keepdims=True) * _sym(rng, M, p) / (2 * p))[1]
    rnd = np.linalg.qr(rng.standard_normal((M, p, p)))[0]
    perm = np.stack([exact[m][rng.permutation(p)] * rng.choice([-1.0, 1.0], p)[:, None] for m in range(M)])
    return {"identity": np.repeat(np.eye(p)[None], M, 0), "exact": exact,
            "perturbed": pert.transpose(0, 2, 1).copy(), "random": rnd, "permuted": perm}


@pytest.mark.parametrize("p,nb2", [(p, 0) for p in (1, 2, 3, 15, 16, 17, 31, 32, 33, 47, 48)]
                         + [(p, 1) for p in (64, 65, 96, 97, 128, 129, 160)])
def test_warm_jacobi_eigenpairs(p, nb2):
    """gg_eigh with Vt_warm: every warm start on every spectrum; the warm buffer returns the new eigenvectors; an exact eigenbasis needs
    one sweep without rotations; vectors = 0 gives the same eigenvalues"""
    A = _spectra_stack(p, p)
    for name, W in _warm_starts(A, p).items():
        r = _twice(lambda: _run_eigh(A, warm=W, nb2=nb2))
        _check_eigpairs(A, r["Vt"], r["D"], "warm")
        assert _same(r["warm"], r["Vt"]), name
        assert r["info"] == 0
        assert (r["sweeps"] >= 1).all() and (r["sweeps"] <= 30).all()
        if name == "exact":
            # LAPACK's eigenvectors leave no off-diagonal cosine above the sweep tolerance -- except inside the
            # 1e-9 cluster and next to the 1e6 offset, where V (A + sigma I) itself rounds at that level
            sw = r["sweeps"][[i for i, k in enumerate(SPECTRA) if k not in ("clustered", "offset")]]
            assert (sw == 1).all(), (name, r["sweeps"])
    # an exactly representable eigenbasis (signed permutation of a diagonal matrix with the same spectra): the warm
    # start diagonalises A exactly, so one sweep without a rotation, whatever the spectrum
    rng = np.random.default_rng(p + 2)
    Ad = np.zeros_like(A)
    Pw = np.zeros_like(A)
    for m in range(len(SPECTRA)):
        perm, sgn = rng.permutation(p), rng.choice([-1.0, 1.0], p)
        Pw[m][np.arange(p), perm] = sgn
        Ad[m][perm, perm] = _ref_eigs(A[m])
    r = _twice(lambda: _run_eigh(Ad, warm=Pw, nb2=nb2))
    _check_eigpairs(Ad, r["Vt"], r["D"], "warm")
    assert (r["sweeps"] == 1).all(), r["sweeps"]
    r0 = _run_eigh(A, nb2=nb2)
    _check_eigpairs(A, r0["Vt"], r0["D"], "cold")
    r1 = _run_eigh(A, nb2=nb2, vectors=0)
    assert _same(r1["D"], r0["D"])


@pytest.mark.parametrize("p,nb2", [(17, 0), (48, 0), (100, 1)])
def test_warm_jacobi_chain_keeps_accuracy(p, nb2):
    """50 warm-chained calls over a slowly drifting matrix, as the ADMM loop makes them: call 50 meets the bound of
    call 1"""
    rng = np.random.default_rng(p)
    M = 2
    A0 = _sym(rng, M, p) + np.linspace(-1, 1, p) * np.eye(p)
    dA = _sym(rng, M, p) * 1e-3
    warm = np.repeat(np.eye(p)[None], M, 0)
    worst = {}
    for t in range(50):
        A = A0 + t * dA
        r = _run_eigh(A, warm=warm, nb2=nb2)
        warm = r["warm"]
        if t in (0, 49):
            worst[t] = _check_eigpairs(A, r["Vt"], r["D"], "chain")
    assert worst[49] <= C_EIG


def test_warm_jacobi_done_problem_untouched():
    """mpp > 1: the matrices of a problem marked done keep A, D and the warm start bitwise"""
    p, K = 20, 3
    rng = np.random.default_rng(1)
    A = _sym(rng, 3 * K, p)
    W = _warm_starts(A, 1)["perturbed"]
    ctrl = _ctrl_np([1.0, 1.0, 1.0], done=[1])
    r = _twice(lambda: _run_eigh(A, warm=W, ctrl=ctrl, mpp=K))
    s = slice(K, 2 * K)
    assert _same(r["Vt"][s], A[s]) and _same(r["warm"][s], W[s]) and (r["D"][s] == FILL).all()
    live = np.r_[0:K, 2 * K:3 * K]
    _check_eigpairs(A[live], r["Vt"][live], r["D"][live], "warm")


@pytest.mark.parametrize("nb2", [32, 64, 128])
@pytest.mark.parametrize("p", [161, 257, 333])
def test_block_jacobi_quad_tol(p, nb2):
    """block Jacobi with the default quadratic-convergence cut-off and without it"""
    rng = np.random.default_rng(p + nb2)
    A = _sym(rng, 2, p)
    A[1] = A[1] @ A[1] / p - 0.5 * np.eye(p)
    for qt in (1e-10, 0.0):
        r = _twice(lambda: _run_eigh(A, nb2=nb2, quad_tol=qt))
        _check_eigpairs(A, r["Vt"], r["D"], "block")
        assert 1 <= r["info"][0] <= 30


# ======================================================================================================================
# 2. stopping test, rho update, pending X scale
# ======================================================================================================================
def _int_split(rng, total, n):
    """n non-negative integers (as doubles) summing to total: any summation order is exact"""
    if not math.isfinite(total):
        v = np.zeros(n)
        v[rng.integers(n)] = total
        return v
    return rng.multinomial(int(total), np.full(n, 1.0 / n)).astype(np.float64)


# (acc0..acc4 totals, rho, pdim, iteration) of the boundary problems; tol = 1, rtol = 0.5
_BOUNDARY = [
    ((0, 0, 0, 100, 4), 0.5, 0.5, 0),      # r = 10 = 10 s: rho doubles
    ((0, 0, 0, 1, 25), 2.0, 0.5, 3),       # s = 10 = 10 r: rho halves
    ((16, 4, 36, 9, 16), 1.0, 1.0, 7),     # r = e_pri = 3, s = e_dual = 4: stops with status 1
    ((16, 4, 36, 9, 16), 1.0, 0.5, 7),     # r = 3 > e_pri = 2.5: goes on
    ((0, 0, 0, math.inf, 1), 1.0, 1.0, 2),  # non-finite: status -1
    ((0, 0, 0, math.nan, 1), 1.0, 1.0, 2),
    ((1, 1, 1, 400, 1), 0.25, 2.0, 5),     # iteration >= hist_cap: nothing written to hist
    ((9, 9, 9, 9, 9), 1.0, 1.0, 1),        # marked done: untouched
]


@pytest.mark.parametrize("nparts", [1, 255, 256, 257, 5000])
@pytest.mark.parametrize("nprob", [1, 3, 2000])
@pytest.mark.parametrize("update_rho", [1, 0])
def test_stop_update_against_host_restatement(nprob, nparts, update_rho):
    from gglasso_b200 import _lib as C
    _l, lib, st = _lib()
    rng = np.random.default_rng(nprob * 7 + nparts)
    hist_cap = 5
    tot = rng.integers(0, 60, (nprob, 5)).astype(np.float64) ** 2
    rho = 2.0 ** rng.integers(-3, 4, nprob)
    pdim = rng.integers(1, 50, nprob).astype(np.float64)
    it = rng.integers(0, 4, nprob)
    done = []
    cases = _BOUNDARY[:nprob] if nprob < len(_BOUNDARY) else _BOUNDARY
    for q, (t, r_, d_, i_) in enumerate(cases):
        tot[q], rho[q], pdim[q], it[q] = t, r_, d_, i_
    if nprob >= len(_BOUNDARY):
        done = [len(_BOUNDARY) - 1]
    parts = np.stack([np.stack([_int_split(rng, tot[q, i], nparts) for i in range(5)], axis=1) for q in range(nprob)])
    ctrl = _ctrl_np(rho, done=done)
    ctrl[:, C.C_ITER] = it
    if nprob > 6:
        ctrl[6, C.C_ITER] = hist_cap + 1
    hist0 = rng.standard_normal((nprob, hist_cap, 5))
    pdev, pdd = _dev(parts), _dev(pdim)

    def run():
        bufs = {"ctrl": _guarded(ctrl.size, ctrl), "hist": _guarded(hist0.size, hist0)}
        rc = lib.gg_stop_update(_p(pdev), nparts, _p(_inner(bufs["ctrl"])), _p(_inner(bufs["hist"])), hist_cap,
                                _p(pdd), 1.0, 0.5, update_rho, nprob, st)
        _l.check(rc, "gg_stop_update")
        return _out(bufs, {"ctrl": ctrl.shape, "hist": hist0.shape})
    got = _twice(run)
    rc, rh = ctrl.copy(), hist0.copy()
    kr.stop_update(parts.sum(axis=1), rc, rh, hist_cap, pdim, 1.0, 0.5, update_rho, C)
    assert _same(got["ctrl"], rc)
    assert _same(got["hist"], rh)
    if nprob >= 3:
        expect = [2.0 * 0.5, 0.5 * 2.0, 1.0] if update_rho else [0.5, 2.0, 1.0]
        assert list(got["ctrl"][:3, C.C_RHO]) == expect
    if nprob >= len(_BOUNDARY):
        g = got["ctrl"]
        assert g[2, C.C_STATUS] == 1 and g[2, C.C_DONE] == 1 and g[3, C.C_DONE] == 0
        assert g[4, C.C_STATUS] == -1 and g[5, C.C_STATUS] == -1 and g[4, C.C_DONE] == 1
        assert g[6, C.C_ITER] == hist_cap + 2 and _same(got["hist"][6], hist0[6])
        assert _same(g[7], ctrl[7]) and _same(got["hist"][7], hist0[7])


@pytest.mark.parametrize("M,p,mpp", [(6, 40, 1), (6, 40, 3), (1500, 64, 1), (1500, 64, 3), (4, 1, 2)])
def test_scale_pending(M, p, mpp):
    """X *= ctrl[xscale] per problem (bitwise), xscale == 1 leaves X alone, and every problem's xscale is reset"""
    from gglasso_b200._lib import C_XSCALE
    _l, lib, st = _lib()
    rng = np.random.default_rng(M + p)
    X = _sym(rng, M, p)
    nprob = M // mpp
    xs = rng.choice([1.0, 0.5, 2.0, 0.3], nprob)
    xs[0] = 1.0
    ctrl = _ctrl_np(np.ones(nprob), xs=xs, done=[nprob - 1])

    def run():
        bufs = {"X": _guarded(X.size, X), "ctrl": _guarded(ctrl.size, ctrl)}
        _l.check(lib.gg_scale_pending(_p(_inner(bufs["X"])), _p(_inner(bufs["ctrl"])), M, p, mpp, st), "scale")
        return _out(bufs, {"X": X.shape, "ctrl": ctrl.shape})
    got = _twice(run)
    xsm = np.repeat(xs, mpp)[:, None, None]
    assert _same(got["X"], np.where(xsm != 1.0, xsm * X, X))
    rc = ctrl.copy()
    rc[:, C_XSCALE] = 1.0
    assert _same(got["ctrl"], rc)


# ======================================================================================================================
# 3. elementwise kernels
# ======================================================================================================================
def _sgl_inputs(M, p, seed, latent):
    rng = np.random.default_rng(seed)
    d = dict(Om=_sym(rng, M, p, 0.3) + 2 * np.eye(p), Omp=_sym(rng, M, p, 0.3), X=_sym(rng, M, p, 0.1),
             L=_sym(rng, M, p, 0.05) if latent else None, lam_mat=np.abs(_sym(rng, M, p, 0.1)),
             rho=rng.uniform(0.5, 2.0, M), pvec=rng.integers(1, p + 1, M).astype(np.int32))
    d["pvec"][0] = p
    return d


@pytest.mark.parametrize("M", [3, 1183, 1184, 1500])
@pytest.mark.parametrize("p", [7, 40, 64])
@pytest.mark.parametrize("variant", ["masked_ragged", "latent"])
def test_prox_sgl(M, p, variant):
    """latent form (C = Theta - X - Omega, X untouched); ragged pvec (padding written, excluded from the partials)
    with an elementwise penalty and rho per matrix; M on both sides of the one-CTA-per-matrix edge"""
    _l, lib, st = _lib()
    latent = variant == "latent"
    d = _sgl_inputs(M, p, M * 100 + p, latent)
    done = [1]
    ctrl = _ctrl_np(d["rho"], done=done)
    n = M * p * p
    nparts = lib.gg_sgl_nparts(p, M)
    assert nparts >= 1
    if p >= 40 and M >= 1184:
        assert _ew_multipass(M, p)
    dv = {k: _dev(d[k]) for k in ("Om", "Omp", "L", "lam_mat")}
    pv = None if latent else _dev(d["pvec"], torch.int32)
    cdev = _dev(ctrl)

    def run():
        bufs = {"X": _guarded(n, d["X"]), "Theta": _guarded(n)}
        if latent:
            bufs["C"] = _guarded(n)
        else:
            bufs["partials"] = _guarded(M * nparts * 5)
        rc = lib.gg_prox_sgl(_p(dv["Om"]), _p(dv["Omp"]), _p(dv["L"]), _p(_inner(bufs["X"])),
                             _p(_inner(bufs["Theta"])), _p(_inner(bufs["C"])) if latent else None, _p(cdev), 0.13,
                             None if latent else _p(dv["lam_mat"]), M, p,
                             None if latent else _p(_inner(bufs["partials"])), _p(pv), st)
        _l.check(rc, "gg_prox_sgl")
        return _out(bufs, {"X": (M, p, p), "Theta": (M, p, p), "C": (M, p, p), "partials": (M, nparts, 5)})
    got = _twice(run)
    assert _same(cdev.cpu().numpy(), ctrl)
    th, o2, parts = kr.prox_sgl(d["Om"], d["Omp"], d["L"], d["X"], 0.13, d["rho"],
                                lam_mat=None if latent else d["lam_mat"], latent=latent,
                                pvec=None if latent else d["pvec"])
    live = np.array([m not in done for m in range(M)])
    assert _same(got["Theta"][live], th[live]) and (got["Theta"][~live] == FILL).all()
    if latent:
        assert _same(got["X"], d["X"])
        assert _same(got["C"][live], o2[live]) and (got["C"][~live] == FILL).all()
    else:
        assert _same(got["X"][live], o2[live]) and _same(got["X"][~live], d["X"][~live])
        assert (got["partials"][~live] == FILL).all()
        for m in np.flatnonzero(live)[:50].tolist() + [M - 1]:
            for i in range(5):
                _check_sums(got["partials"][m, :, i], parts[m, i], "prox_sgl_partials")


@pytest.mark.parametrize("Mblk", [1, 2, 3, 5, 7])
@pytest.mark.parametrize("nb", [1, 2, 9, 33, 70])
@pytest.mark.parametrize("latent", [False, True])
def test_prox_fsgl(Mblk, nb, latent):
    """block norms (fsgl_block_norm_kernel) over several CTAs with a partial last one, latent and not, bitwise against the kernel-order
    reference; Mblk = 1 within 1 ulp of gg_prox_sgl"""
    _l, lib, st = _lib()
    p, M = Mblk * nb, 3
    d = _sgl_inputs(M, p, Mblk * 1000 + nb, latent)
    ctrl = _ctrl_np(d["rho"], done=[1])
    n = M * p * p
    nparts = lib.gg_sgl_nparts(p, M)
    dv = {k: _dev(d[k]) for k in ("Om", "Omp", "L")}
    cdev = _dev(ctrl)

    def run(fsgl=True):
        bufs = {"X": _guarded(n, d["X"]), "Theta": _guarded(n)}
        if latent:
            bufs["C"] = _guarded(n)
        else:
            bufs["partials"] = _guarded(M * nparts * 5)
        args = (_p(dv["Om"]), _p(dv["Omp"]), _p(dv["L"]), _p(_inner(bufs["X"])), _p(_inner(bufs["Theta"])),
                _p(_inner(bufs["C"])) if latent else None, _p(cdev), 0.21)
        parts = None if latent else _p(_inner(bufs["partials"]))
        if fsgl:
            bufs["blk"] = _guarded(M * nb * nb)
            rc = lib.gg_prox_fsgl(*args, Mblk, M, p, parts, _p(_inner(bufs["blk"])), st)
        else:
            rc = lib.gg_prox_sgl(*args, None, M, p, parts, None, st)
        _l.check(rc, "gg_prox_fsgl")
        return _out(bufs, {"X": (M, p, p), "Theta": (M, p, p), "C": (M, p, p), "partials": (M, nparts, 5),
                           "blk": (M * nb * nb,)})
    got = _twice(run)
    nrm = kr.block_norms(d["Om"] + (d["L"] if latent else 0.0) + d["X"], Mblk)
    up = np.triu(np.ones((nb, nb), dtype=bool), 1)
    blk = got["blk"].reshape(M, nb, nb)
    assert _same(blk[0][up], nrm[0][up]) and _same(blk[2][up], nrm[2][up]) and (blk[1] == FILL).all()
    th, o2, parts = kr.prox_fsgl(d["Om"], d["Omp"], d["L"], d["X"], 0.21, d["rho"], Mblk, latent=latent)
    live = [0, 2]
    assert _same(got["Theta"][live], th[live]) and (got["Theta"][1] == FILL).all()
    if latent:
        assert _same(got["C"][live], o2[live]) and _same(got["X"], d["X"])
    else:
        assert _same(got["X"][live], o2[live]) and _same(got["X"][1], d["X"][1])
        for m in live:
            for i in range(5):
                _check_sums(got["partials"][m, :, i], parts[m, i], "prox_fsgl_partials")
    for m in live:
        A = d["Om"][m] + (d["L"][m] if latent else 0.0) + d["X"][m]
        ref = kr.prox_sum_frob(A, Mblk, (1.0 / d["rho"][m]) * 0.21)
        err = np.abs(got["Theta"][m] - ref).max() / max(np.abs(ref).max(), 1e-300)
        _note("fsgl_vs_prox_sum_frob", err)
        assert err < 1e-14
    if Mblk == 1:
        sgl = run(fsgl=False)
        np.testing.assert_array_max_ulp(got["Theta"][live], sgl["Theta"][live], maxulp=1)


def test_prox_fsgl_rejects_indivisible_blocks():
    _l, lib, st = _lib()
    z = torch.zeros(2 * 10 * 10, dtype=torch.float64, device="cuda")
    c = _dev(_ctrl_np([1.0, 1.0]))
    assert lib.gg_prox_fsgl(_p(z), _p(z), None, _p(z), _p(z), None, _p(c), 0.1, 3, 2, 10, _p(z), _p(z), st) == -1


@pytest.mark.parametrize("sgl_order", [0, 1])
@pytest.mark.parametrize("with_L", [False, True])
@pytest.mark.parametrize("M,mpp", [(6, 1), (6, 3), (1500, 1), (1500, 3)])
def test_dual_update(sgl_order, with_L, M, mpp):
    _l, lib, st = _lib()
    p = 40
    assert _ew_multipass(M, p) == (M == 1500)
    rng = np.random.default_rng(M + 10 * sgl_order + with_L)
    X, Om, Omp, Th = (_sym(rng, M, p, s) for s in (0.1, 1.0, 1.0, 0.7))
    L = _sym(rng, M, p, 0.05) if with_L else None
    nprob = M // mpp
    ctrl = _ctrl_np(np.ones(nprob), done=[1])
    nparts = lib.gg_sgl_nparts(p, M)
    dv = [_dev(a) for a in (Om, Omp, Th, L)]
    cdev = _dev(ctrl)

    def run():
        bufs = {"X": _guarded(X.size, X), "partials": _guarded(M * nparts * 5)}
        rc = lib.gg_dual_update(_p(_inner(bufs["X"])), *[_p(a) for a in dv], _p(cdev), M, p, mpp, sgl_order,
                                _p(_inner(bufs["partials"])), st)
        _l.check(rc, "gg_dual_update")
        return _out(bufs, {"X": X.shape, "partials": (M, nparts, 5)})
    got = _twice(run)
    assert _same(cdev.cpu().numpy(), ctrl)
    xn, parts = kr.dual_update(X, Om, Omp, Th, L, sgl_order)
    live = np.repeat(np.arange(nprob) != 1, mpp)
    assert _same(got["X"][live], xn[live]) and _same(got["X"][~live], X[~live])
    assert (got["partials"][~live] == FILL).all()
    for m in np.flatnonzero(live)[:40]:
        for i in range(5):
            _check_sums(got["partials"][m, :, i], parts[m, i], "dual_update_partials")


@pytest.mark.parametrize("with_L", [False, True])
@pytest.mark.parametrize("with_nk", [False, True])
@pytest.mark.parametrize("M,mpp", [(6, 1), (6, 3), (1500, 3)])
def test_build_w(with_L, with_nk, M, mpp):
    """W = Theta - L - xs X - (n_k/rho) S with a pending X scale folded in and stored; ctrl is not written"""
    _l, lib, st = _lib()
    p = 40
    rng = np.random.default_rng(M + 2 * with_L + with_nk)
    Th, X, S = (_sym(rng, M, p, s) for s in (1.0, 0.2, 1.0))
    L = _sym(rng, M, p, 0.05) if with_L else None
    nk = rng.uniform(20, 200, M) if with_nk else None
    nprob = M // mpp
    rho = rng.uniform(0.3, 3.0, nprob)
    xs = rng.choice([1.0, 0.5, 2.0, 0.7], nprob)
    ctrl = _ctrl_np(rho, xs=xs, done=[1])
    dv = [_dev(a) for a in (Th, L)]
    sd, nkd, cdev = _dev(S), _dev(nk), _dev(ctrl)

    def run():
        bufs = {"X": _guarded(X.size, X), "W": _guarded(X.size)}
        rc = lib.gg_build_w(_p(dv[0]), _p(dv[1]), _p(_inner(bufs["X"])), _p(sd), _p(nkd), _p(cdev), M, p, mpp,
                            _p(_inner(bufs["W"])), st)
        _l.check(rc, "gg_build_w")
        return _out(bufs, {"X": X.shape, "W": X.shape})
    got = _twice(run)
    assert _same(cdev.cpu().numpy(), ctrl)
    w, xv = kr.build_w(Th, L, X, S, nk, np.repeat(rho, mpp), np.repeat(xs, mpp))
    live = np.repeat(np.arange(nprob) != 1, mpp)
    assert _same(got["W"][live], w[live]) and (got["W"][~live] == FILL).all()
    assert _same(got["X"][live], xv[live]) and _same(got["X"][~live], X[~live])


def _ext_case(K, seed, latent):
    rng = np.random.default_rng(seed)
    pvec = [200, 137] if K == 2 else [37, 150, 1, 90, 64]
    P = max(pvec)

    def padded(scale):
        A = _sym(rng, K, P, scale)                         # padding: values the kernels must keep out of the sums
        for k, pk in enumerate(pvec):
            A[k, :pk, :pk] = _sym(rng, 1, pk, scale)[0]
        return A
    d = dict(Om=padded(0.5), X0=padded(0.1), Lam=padded(0.3), X1=padded(0.1), Omp=padded(0.5), Lamp=padded(0.3),
             L=padded(0.05) if latent else None, lam1=rng.uniform(0.05, 0.3, K), G=kr.ext_groups(pvec, rng),
             pvec=np.array(pvec, dtype=np.int32), rho=1.7, lambda2=0.09)
    return d, P


@pytest.mark.parametrize("K", [2, 5])
@pytest.mark.parametrize("latent", [False, True])
@pytest.mark.parametrize("done", [False, True])
def test_ext_kernels(K, latent, done):
    """gg_ext_theta, gg_ext_lambda and gg_ext_dual on ragged padded stacks against the kernel-order references:
    Lambda is Theta + X1 except at the group members, written in both triangles"""
    _l, lib, st = _lib()
    d, P = _ext_case(K, K * 10 + latent, latent)
    ctrl = _ctrl_np([d["rho"]], done=[0] if done else [])
    n = K * P * P
    nparts = K * lib.gg_sgl_nparts(P, K)
    dv = {k: _dev(d[k]) for k in ("Om", "X0", "Lam", "X1", "Omp", "Lamp", "L", "lam1")}
    Gd, pv, cdev = _dev(d["G"], torch.int32), _dev(d["pvec"], torch.int32), _dev(ctrl)
    Lg = d["G"].shape[1]
    sh = (K, P, P)

    def run():
        b = {"Theta": _guarded(n), "Lam": _guarded(n), "X0": _guarded(n, d["X0"]), "X1": _guarded(n, d["X1"]),
             "partials": _guarded(nparts * 5)}
        if latent:
            b["C"] = _guarded(n)
        _l.check(lib.gg_ext_theta(_p(dv["Om"]), _p(dv["L"]), _p(dv["X0"]), _p(dv["Lam"]), _p(dv["X1"]),
                                  _p(dv["lam1"]), _p(cdev), K, P, _p(_inner(b["Theta"])),
                                  _p(_inner(b["C"])) if latent else None, st), "gg_ext_theta")
        _l.check(lib.gg_ext_lambda(_p(_inner(b["Theta"])), _p(dv["X1"]), _p(Gd), Lg, K, P, d["lambda2"], _p(cdev),
                                   _p(_inner(b["Lam"])), st), "gg_ext_lambda")
        _l.check(lib.gg_ext_dual(_p(_inner(b["X0"])), _p(_inner(b["X1"])), _p(dv["Om"]), _p(dv["Omp"]),
                                 _p(_inner(b["Theta"])), _p(dv["L"]), _p(_inner(b["Lam"])), _p(dv["Lamp"]), _p(cdev),
                                 _p(pv), K, P, _p(_inner(b["partials"])), st), "gg_ext_dual")
        return _out(b, {"Theta": sh, "Lam": sh, "X0": sh, "X1": sh, "C": sh, "partials": (K, nparts // K, 5)})
    got = _twice(run)
    assert _same(cdev.cpu().numpy(), ctrl)
    if done:
        for k in ("Theta", "Lam", "partials") + (("C",) if latent else ()):
            assert (got[k] == FILL).all(), k
        assert _same(got["X0"], d["X0"]) and _same(got["X1"], d["X1"])
        return
    th, C = kr.ext_theta(d["Om"], d["L"], d["X0"], d["Lam"], d["X1"], d["lam1"], d["rho"])
    assert _same(got["Theta"], th)
    if latent:
        assert _same(got["C"], C)
    lam = kr.ext_lambda(th, d["X1"], d["G"], d["lambda2"], d["rho"])
    assert _same(got["Lam"], lam)
    member = np.zeros(sh, dtype=bool)
    for k in range(K):
        g = d["G"][:, d["G"][0, :, k] >= 0, k]
        member[k, g[0], g[1]] = member[k, g[1], g[0]] = True
    assert _same(got["Lam"][~member], (th + d["X1"])[~member])
    x0, x1, parts = kr.ext_dual(d["X0"], d["X1"], d["Om"], d["Omp"], th, d["L"], lam, d["Lamp"], d["pvec"])
    assert _same(got["X0"], x0) and _same(got["X1"], x1)
    for k in range(K):
        for i in range(5):
            _check_sums(got["partials"][k, :, i], parts[k, i], "ext_dual_partials")


@pytest.mark.parametrize("total", [1, 3 * 37 * 37, 148 * 16 * 256 * 2 + 77])
@pytest.mark.parametrize("with_L", [False, True])
def test_add3(total, with_L):
    _l, lib, st = _lib()
    rng = np.random.default_rng(total)
    Om, L, X = rng.standard_normal(total), rng.standard_normal(total), rng.standard_normal(total)
    L = L if with_L else None
    dv = [_dev(a) for a in (Om, L, X)]

    def run():
        b = {"V": _guarded(total)}
        _l.check(lib.gg_add3(*[_p(a) for a in dv], _p(_inner(b["V"])), total, st), "gg_add3")
        return _out(b, {"V": (total,)})
    assert _same(_twice(run)["V"], kr.add3(Om, L, X))


# ======================================================================================================================
# 4. reductions and checks
# ======================================================================================================================
@pytest.mark.parametrize("reg", [-1, 0, 1])
@pytest.mark.parametrize("K", [1, 3, 20, 90])
@pytest.mark.parametrize("p", [1, 17, 257, 1000])
def test_objective(reg, K, p):
    """<Omega,S> and P(Theta) against exact sums; only the strict upper triangle of Theta enters P (the rest is
    seeded with garbage that would dominate it)"""
    if K == 90 and p == 1000:
        pytest.skip("720 MB per array; K = 90 is covered at p <= 257 and p = 1000 at K <= 20")
    _l, lib, st = _lib()
    rng = np.random.default_rng(K * 1000 + p)
    Om, S = _sym(rng, K, p), _sym(rng, K, p)
    Th = _sym(rng, K, p, 0.3)
    lower = np.tril(np.ones((p, p), dtype=bool))
    Th[:, lower] = 1e30
    nparts = lib.gg_objective_nparts(p)
    dv = [_dev(a) for a in (Om, S, Th)]

    def run():
        b = {"partials": _guarded(2 * nparts)}
        _l.check(lib.gg_objective(*[_p(a) for a in dv], 0.3, 0.2, reg, K, p, _p(_inner(b["partials"])), st),
                 "gg_objective")
        return _out(b, {"partials": (nparts, 2)})
    got = _twice(run)["partials"]
    ip, ip_abs, P = kr.objective_parts(Om, S, Th, 0.3, 0.2, reg)
    _check_sums(got[:, 0], ip, "objective_inner", abs_ref=ip_abs)
    if reg < 0 or p == 1:
        assert (got[:, 1] == 0).all()
    else:
        _check_sums(got[:, 1], P, "objective_penalty")


@pytest.mark.parametrize("p", [37, 257])
def test_asym_max(p):
    _l, lib, st = _lib()
    rng = np.random.default_rng(p)
    M = 4
    A = _sym(rng, M, p)
    spots = [(0, p - 1), (p - 2, p - 1), (p // 2, p // 2 + 3)]
    want = np.zeros(M)
    for m, (i, j) in enumerate(spots):
        A[m, j, i] = A[m, i, j] + 1e-7 * (m + 1)
        want[m] = abs(A[m, i, j] - A[m, j, i])
    nparts = lib.gg_sgl_nparts(p, M)
    ad = _dev(A)

    def run():
        b = {"out": _guarded(M * nparts)}
        _l.check(lib.gg_asym_max(_p(ad), M, p, _p(_inner(b["out"])), st), "gg_asym_max")
        return _out(b, {"out": (M, nparts)})
    got = _twice(run)["out"]
    assert _same(got.max(axis=1), want)


def _run_gersh(A):
    _l, lib, st = _lib()
    M, p, _ = A.shape
    ws_bytes = int(lib.gg_eigh_workspace_bytes(M, p))
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    ad = _dev(A)

    def run():
        b = {"out": _guarded(M)}
        _l.check(lib.gg_gershgorin_min(_p(ad), M, p, _p(ws), ws_bytes, _p(_inner(b["out"])), st), "gg_gershgorin")
        return _out(b, {"out": (M,)})
    return _twice(run)["out"]


@pytest.mark.parametrize("p", [1, 5, 17, 48, 49, 100, 257])
def test_gershgorin_min_against_exact_bound(p):
    """with the workspace of Eigh(M, p), as the engine calls it: a lower bound, and tight to a few p u sum |a_ij|"""
    rng = np.random.default_rng(p)
    M = 5
    A = _sym(rng, M, p) + np.linspace(0, 3 * p, M)[:, None, None] * np.eye(p)
    got = _run_gersh(A)
    exact = kr.gershgorin_exact(A)
    for m in range(M):
        assert Fraction(got[m]) <= exact[m]
        slack = float(exact[m] - Fraction(got[m])) / (p * EPS * np.abs(A[m]).sum(axis=1).max())
        _note("gershgorin_slack_p_u_rowsum", slack)
        assert slack <= 4.0


def _rdown(fr):
    f = float(fr)
    return f if Fraction(f) <= fr else float(np.nextafter(f, -np.inf))


@pytest.mark.parametrize("p", [33, 100, 162])
def test_gershgorin_certificate_is_sound(p):
    """rows whose diagonal equals the rounded-down sum of the off-diagonal magnitudes (and a few ulps above it):
    whenever the kernel returns a positive bound the exact bound is positive.  Summing the diagonal into the row sum
    and subtracting it again gave positive bounds for rows whose exact bound was negative."""
    M = 64
    rng = np.random.default_rng(p)
    A = np.zeros((M, p, p))
    for m in range(M):
        a = rng.uniform(-0.01, 0.01, (p, p))
        a = (a + a.T) / 2
        i = int(rng.integers(p))
        col = -rng.uniform(0.1, 1.0, p)
        a[i, :], a[:, i] = col, col
        np.fill_diagonal(a, 10.0 * p)
        S = sum(Fraction(abs(x)) for j, x in enumerate(a[i].tolist()) if j != i)
        d = _rdown(S)
        for _ in range(m % 4):
            d = float(np.nextafter(d, np.inf))
        a[i, i] = d
        A[m] = a
    got = _run_gersh(A)
    exact = kr.gershgorin_exact(A)
    for m in range(M):
        if got[m] > 0:
            assert exact[m] > 0, (m, got[m], float(exact[m]))
        assert Fraction(got[m]) <= exact[m]


@pytest.mark.parametrize("p", [5, 64, 161])
@pytest.mark.parametrize("mpp", [1, 2])
def test_recon_rho_from_ctrl(p, mpp):
    """gg_recon with bnum = NULL and rho read from ctrl per problem (a done problem's output untouched), modes 0/1/2;
    extends test_recon_modes"""
    _l, lib, st = _lib()
    rng = np.random.default_rng(p + mpp)
    M = 4
    A = _sym(rng, M, p)
    D, Q = np.linalg.eigh(A)
    Vt = np.ascontiguousarray(Q.transpose(0, 2, 1))
    nprob = M // mpp
    rho = rng.uniform(0.3, 3.0, nprob)
    ctrl = _ctrl_np(rho, done=[1])
    vd, dd, cdev = _dev(Vt), _dev(D), _dev(ctrl)
    fs = {0: lambda d, b: 0.5 * (np.sqrt(d * d + 4 * b) + d), 1: lambda d, b: np.maximum(d - b, 0), 2: lambda d, b: d}
    for mode, f in fs.items():
        def run():
            b = {"Out": _guarded(A.size)}
            _l.check(lib.gg_recon(_p(vd), _p(dd), None, _p(cdev), mpp, mode, M, p, _p(_inner(b["Out"])), st), "recon")
            return _out(b, {"Out": A.shape})
        got = _twice(run)["Out"]
        for m in range(M):
            q = m // mpp
            if q == 1:
                assert (got[m] == FILL).all()
                continue
            ref = (Q[m] * f(D[m], 1.0 / rho[q])) @ Q[m].T
            err = np.linalg.norm(got[m] - ref) / max(np.linalg.norm(ref), 1e-300)
            _note("recon_rel_frob", err)
            assert err < 1e-12, (mode, m, err)
            assert np.array_equal(got[m], got[m].T)
