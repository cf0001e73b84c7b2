"""Device-resident ADMM loop shared by ADMM_MGL / ADMM_SGL / block_SGL.

torch is used for device memory, streams and host<->device copies only; every arithmetic step
of the iteration is a hand-written sm_100a kernel reached through the C ABI (_lib.py).
One iteration (reference: src/gglasso/solver/admm_solver.py:172-246) is

    gg_build_w -> gg_eigh -> gg_recon(phi+) -> gg_prox_* [-> gg_eigh -> gg_recon(shrink) -> gg_dual_update]
    -> gg_stop_update

and rho, the pending dual rescale, the residual history and the done flag stay on the device,
so the host only polls the done flag every ``check_every`` iterations.
"""
import ctypes
import os
import time

import numpy as np
import torch

from . import _lib
from ._lib import CTRL_STRIDE, HIST_STRIDE, NPART, C_DONE, C_ITER, C_RHO, C_XSCALE, C_STATUS, C_LAM1, C_LAM2


# largest K of the fused tile-pair MGL prox (K x 272 doubles of shared memory per CTA <= 200 KB)
K_TILE_MAX = 90


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def control_block(nprob, rho, lambdas=None):
    """fresh host control block of ``nprob`` problems (float64, (nprob, CTRL_STRIDE)): rho, no pending dual rescale and,
    for MGL, ``lambdas`` = (lambda1, lambda2), each a scalar or one value per problem."""
    ctrl = np.zeros((nprob, CTRL_STRIDE))
    ctrl[:, C_RHO] = rho
    ctrl[:, C_XSCALE] = 1.0
    if lambdas is not None:
        ctrl[:, C_LAM1], ctrl[:, C_LAM2] = lambdas
    return ctrl


def boyd_status(ctrl, hist):
    """the reference's status of one problem after the 'boyd' loop, and its residual series max(r_t, s_t).
    ``ctrl``: the problem's control block row; ``hist``: its residual history, one row per iteration."""
    n = int(ctrl[C_ITER])
    r, s, e_pri, e_dual = hist[n - 1, :4]
    if ctrl[C_DONE] != 0:
        status = "optimal"
    elif r <= e_pri:
        status = "primal optimal"
    elif s <= e_dual:
        status = "dual optimal"
    else:
        status = "max iterations reached"
    return status, np.maximum(hist[:n, 0], hist[:n, 1])


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def require_cuda():
    if not torch.cuda.is_available():
        raise _lib.GGLassoB200Error("gglasso_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
    return torch.device("cuda", torch.cuda.current_device())


def to_dev(a, dev):
    """numpy (or torch) -> contiguous FP64 device tensor (copy).

    Large host arrays go through pinned staging buffers filled by several host threads at once (numpy's copy releases
    the GIL; a single thread moves ~5-8 GB/s, far below the PCIe link), each thread feeding its own CUDA stream."""
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=torch.float64, copy=True).contiguous()
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.nbytes < (8 << 20):
        return torch.from_numpy(a).to(dev, non_blocking=False)
    dev = torch.device(dev)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    src = torch.from_numpy(a)
    if src.is_pinned():             # caller's array is already page-locked: one DMA, no staging copy
        out = torch.empty(a.shape, dtype=torch.float64, device=dev)
        out.copy_(src, non_blocking=True)         # (stream ordered; every solver call synchronises before it returns)
        return out
    with _H2D_LOCK:
        return _to_dev_staged(a, dev)


def _to_dev_staged(a, dev):
    out = torch.empty(a.shape, dtype=torch.float64, device=dev)
    src = torch.from_numpy(a).view(-1)
    dst = out.view(-1)
    n = src.numel()
    lanes = _h2d_lanes(dev)
    nl = len(lanes)
    per = (n + nl - 1) // nl
    main = torch.cuda.current_stream(dev)
    start = torch.cuda.Event()
    start.record(main)                                 # `out` was allocated on the main stream

    def work(w):
        lo0, hi0 = w * per, min(n, (w + 1) * per)
        bufs, evs, stream = lanes[w]
        ce = bufs[0].numel()
        torch.cuda.set_device(dev)
        stream.wait_event(start)
        with torch.cuda.stream(stream):
            for i, lo in enumerate(range(lo0, hi0, ce)):
                hi = min(hi0, lo + ce)
                evs[i & 1].synchronize()               # previous H2D out of this buffer has finished
                bufs[i & 1][:hi - lo].copy_(src[lo:hi])
                dst[lo:hi].copy_(bufs[i & 1][:hi - lo], non_blocking=True)
                evs[i & 1].record(stream)
            done = torch.cuda.Event()
            done.record(stream)
        return done

    for done in _pool().map(work, range(nl)):
        main.wait_event(done)
    return out


_STAGE = {}
_H2D_LOCK = __import__("threading").Lock()
_H2D_THREADS = max(1, _env_int("GG_H2D_THREADS", 4))


def _pool():
    if "pool" not in _STAGE:
        from concurrent.futures import ThreadPoolExecutor
        _STAGE["pool"] = ThreadPoolExecutor(max_workers=_H2D_THREADS, thread_name_prefix="gg_h2d")
    return _STAGE["pool"]


def _h2d_lanes(dev, chunk_bytes=16 << 20):
    """per device: one lane per copy thread = (two pinned staging buffers, their events, a CUDA stream)"""
    key = ("lanes", dev.index)
    if key not in _STAGE:
        lanes = []
        for _ in range(_H2D_THREADS):
            bufs = [torch.empty(chunk_bytes // 8, dtype=torch.float64, pin_memory=True) for _ in range(2)]
            evs = [torch.cuda.Event(), torch.cuda.Event()]
            lanes.append((bufs, evs, torch.cuda.Stream(device=dev)))
        _STAGE[key] = lanes
    return _STAGE[key]


def warmup():
    """one-time process initialisation (library load, pinned staging buffers); optional."""
    _lib.load()
    dev = require_cuda()
    _h2d_lanes(dev)
    _pool()


def to_host(t):
    """device tensor -> fresh numpy array.  The array lives in page-locked memory from torch's caching host allocator
    (returned to the cache when the caller drops the array), so the device->host DMA writes the result directly --
    no staging buffer and no host-side memcpy; repeated calls reuse the pinned blocks."""
    t = t.contiguous()
    if t.numel() * 8 <= (1 << 20):
        return t.cpu().numpy()
    host = torch.empty(t.shape, dtype=torch.float64, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return host.numpy()


def to_host_many(tensors):
    """several device tensors -> numpy arrays with all copies in flight before one synchronisation"""
    hosts = []
    for t in tensors:
        t = t.contiguous()
        h = torch.empty(t.shape, dtype=torch.float64, pin_memory=True)
        h.copy_(t, non_blocking=True)
        hosts.append(h)
    if tensors:
        torch.cuda.current_stream(tensors[0].device).synchronize()
    return [h.numpy() for h in hosts]


_DEBUG_KEEP_INPUT = bool(int(os.environ.get("GG_DEBUG_KEEP_INPUT", "0")))
_DEBUG_BUFFERS = []


def _debug_check(st, it, where, **arrays):
    """diagnostics (GG_DEBUG_KEEP_INPUT=1): first non-finite array of an iteration -> exception naming it"""
    torch.cuda.current_stream().synchronize()
    for name, a in arrays.items():
        fin = torch.isfinite(a.reshape(a.shape[0], -1)).all(dim=1)
        if not bool(fin.all()):
            bad = torch.nonzero(~fin).flatten().tolist()
            raise FloatingPointError(f"non-finite {name} {where}, iteration {it}, matrices {bad}, "
                                     f"ctrl={st.ctrl[0, :9].tolist()}")


class Eigh:
    """workspace + call wrapper for gg_eigh / gg_recon on (M,p,p) stacks."""

    def __init__(self, M, p, dev):
        self.lib = _lib.load()
        self.M, self.p = M, p
        self.ws_bytes = int(self.lib.gg_eigh_workspace_bytes(M, p))
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.D = torch.empty((M, p), dtype=torch.float64, device=dev)
        self.info = (ctypes.c_int * 4)()
        self.nb2 = _env_int("GG_BLOCK_NB2", 0)
        self.quad_tol = float(os.environ.get("GG_QUAD_TOL", "1e-10"))
        self.sweeps = []

    def eigh(self, A, ctrl=None, mpp=1, vectors=1, stream=0, warm=None):
        if _DEBUG_KEEP_INPUT:
            # diagnostics (GG_DEBUG_KEEP_INPUT=1): keep a host copy of the last input of every workspace so that a
            # failing decomposition can be replayed (scripts/gpu_replay_eigh.py)
            if not hasattr(self, "_dbg"):
                self._dbg = torch.empty(A.shape, dtype=A.dtype, pin_memory=True)
                _DEBUG_BUFFERS.append((self, self._dbg))
            torch.cuda.current_stream().synchronize()
            self._dbg.copy_(A)
            self._dbg_args = (mpp, vectors, None if ctrl is None else ctrl.detach().cpu().numpy().copy())
        rc = self.lib.gg_eigh(_p(A), _p(self.D), self.M, self.p, _p(ctrl), mpp, _p(self.ws), self.ws_bytes,
                              vectors, self.nb2, 0.0, 0, self.quad_tol, self.info, _p(warm), stream)
        _lib.check(rc, "gg_eigh")
        self.sweeps.append(self.info[0])
        return self.D

    def recon(self, Vt, out, mode, bnum=None, ctrl=None, mpp=1, stream=0):
        rc = self.lib.gg_recon(_p(Vt), _p(self.D), _p(bnum), _p(ctrl), mpp, mode, self.M, self.p, _p(out), stream)
        _lib.check(rc, "gg_recon")
        return out


def eigh(A, nb2=None):
    """Public helper: batched symmetric eigendecomposition of (M,p,p) / (p,p) numpy input on the GPU.

    Returns (D ascending, Q with eigenvectors as columns) like np.linalg.eigh.
    ``nb2`` in {32, 64, 128} forces the block-Jacobi path for p > 160 (default: tridiagonal D&C path).
    """
    dev = require_cuda()
    A = np.asarray(A, dtype=np.float64)
    single = A.ndim == 2
    At = to_dev(A[None] if single else A, dev)
    M, p, _ = At.shape
    e = Eigh(M, p, dev)
    if nb2 is not None:
        e.nb2 = nb2
    D = e.eigh(At, stream=torch.cuda.current_stream().cuda_stream)
    D, order = torch.sort(D, dim=1)
    Vt = torch.gather(At, 1, order[:, :, None].expand(M, p, p))
    Q = Vt.transpose(1, 2).contiguous()
    D, Q = D.cpu().numpy(), Q.cpu().numpy()
    return (D[0], Q[0]) if single else (D, Q)


class AdmmState:
    """Device buffers of one batched ADMM run: M matrices, ``mpp`` per problem.  ``lambdas`` (MGL): (lambda1, lambda2)
    for the control block, where the MGL kernels read them (see control_block)."""

    def __init__(self, S, Omega_0, Theta_0, X_0, mpp, rho, max_iter, latent, nk=None, mu=None, lam_mat=None,
                 pvec=None, lambdas=None):
        self.lib = _lib.load()
        self.dev = dev = require_cuda()
        self.S = to_dev(S, dev)
        self.M, self.p, _ = self.S.shape
        self.mpp = mpp
        self.nprob = self.M // mpp
        self.latent = latent
        self.Omega = to_dev(Omega_0, dev)
        self.Omega_new = torch.empty_like(self.Omega)
        self._bufA, self._bufB = self.Omega, self.Omega_new
        # defaults of the reference (admm_solver.py:143-146) are formed on the device: no extra uploads
        self.Theta = self.Omega.clone() if Theta_0 is None else to_dev(Theta_0, dev)
        self.X = torch.zeros_like(self.S) if X_0 is None else to_dev(X_0, dev)
        self.L = torch.zeros_like(self.S) if latent else None
        self.W = torch.empty_like(self.S)
        self.eig = Eigh(self.M, self.p, dev)
        # warm start of the small-matrix eigensolver: previous eigenvectors of W (and of C when latent)
        self.warm_w = self.warm_c = None
        if self.p <= 48 and os.environ.get("GG_NO_WARM", "0") != "1":
            eye = torch.eye(self.p, dtype=torch.float64, device=dev)
            self.warm_w = eye.repeat(self.M, 1, 1).contiguous()
            self.warm_c = self.warm_w.clone() if latent else None
        self.nk = None if nk is None else to_dev(nk, dev)
        self.mu = None if mu is None else to_dev(mu, dev)
        self.lam_mat = None if lam_mat is None else to_dev(lam_mat, dev)
        self.ctrl = to_dev(control_block(self.nprob, rho, lambdas), dev)
        self.hist_cap = max_iter
        self.hist = torch.zeros((self.nprob, max_iter, HIST_STRIDE), dtype=torch.float64, device=dev)
        p = self.p
        self.pvec = None
        if pvec is None:
            self.pdim = to_dev(np.full(self.nprob, mpp * ((p ** 2 + p) / 2)), dev)
        else:                               # ragged batch of independent problems, problem q padded from p_q to p
            pv = np.asarray(pvec, dtype=np.int64)
            self.pvec = torch.from_numpy(pv.astype(np.int32)).to(dev)
            self.pdim = to_dev(mpp * ((pv ** 2 + pv) / 2.0), dev)
        self.stream = torch.cuda.current_stream().cuda_stream

    def reset(self, Omega_0, Theta_0=None, X_0=None, rho=1.0, lambdas=None):
        """re-arm the state for another solve of the same shape on the same buffers (lambda grids).
        ``lambdas`` = (lambda1, lambda2) go into the control block."""
        if self.Omega is not self._bufA:
            self.Omega, self.Omega_new = self._bufA, self._bufB
        self.Omega.copy_(Omega_0 if isinstance(Omega_0, torch.Tensor) else to_dev(Omega_0, self.dev))
        if Theta_0 is None:
            self.Theta.copy_(self.Omega)
        else:
            self.Theta.copy_(Theta_0 if isinstance(Theta_0, torch.Tensor) else to_dev(Theta_0, self.dev))
        if X_0 is None:
            self.X.zero_()
        else:
            self.X.copy_(X_0 if isinstance(X_0, torch.Tensor) else to_dev(X_0, self.dev))
        if self.L is not None:
            self.L.zero_()
        self.ctrl.copy_(torch.from_numpy(control_block(self.nprob, rho, lambdas)), non_blocking=False)
        self.hist.zero_()

    # -- one Omega step: W build, eigh, phi+ reconstruction into Omega_new -----------------
    def omega_step(self, upper=False):
        lib, st = self.lib, self.stream
        if upper:       # upper triangles only (see run_admm): the tridiagonal eigensolver reads nothing else of W
            _lib.check(lib.gg_build_w_upper_batch(_p(self.Theta), _p(self.X), _p(self.S), _p(self.nk), _p(self.ctrl),
                                                  self.mpp, self.p, self.nprob, _p(self.W), st), "gg_build_w_upper")
        else:
            _lib.check(lib.gg_build_w(_p(self.Theta), _p(self.L), _p(self.X), _p(self.S), _p(self.nk), _p(self.ctrl),
                                      self.M, self.p, self.mpp, _p(self.W), st), "gg_build_w")
        self.eig.eigh(self.W, ctrl=self.ctrl, mpp=self.mpp, stream=st, warm=self.warm_w)
        self.eig.recon(self.W, self.Omega_new, 0, bnum=self.nk, ctrl=self.ctrl, mpp=self.mpp, stream=st)

    def l_step(self):
        """latent: W holds C = Theta - X - Omega; L = V max(D - mu/rho, 0) V^T."""
        st = self.stream
        self.eig.eigh(self.W, ctrl=self.ctrl, mpp=self.mpp, stream=st, warm=self.warm_c)
        self.eig.recon(self.W, self.L, 1, bnum=self.mu, ctrl=self.ctrl, mpp=self.mpp, stream=st)

    def mirror(self):
        """fill the lower triangles of Theta and X from the upper ones (after iterations that ran on the upper
        triangles only)"""
        _lib.check(self.lib.gg_mirror_upper(_p(self.Theta), _p(self.X), self.M, self.p, self.stream), "gg_mirror_upper")

    def swap(self):
        self.Omega, self.Omega_new = self.Omega_new, self.Omega

    def final_omega(self, iters):
        """Omega of problem q lives in the buffer written by its last *executed* iteration (kernels are
        no-ops once a problem is done, while the host keeps alternating the two buffers)."""
        bufs = (self._bufA, self._bufB)            # iteration t (1-based) writes bufs[t % 2]
        it = torch.as_tensor(np.asarray(iters), device=self.dev).repeat_interleave(self.mpp)
        odd = (it % 2 == 1).reshape(-1, 1, 1)
        return torch.where(odd, bufs[1], bufs[0])

    def read_ctrl(self):
        return self.ctrl.cpu().numpy()

    def finish_x(self):
        _lib.check(self.lib.gg_scale_pending(_p(self.X), _p(self.ctrl), self.M, self.p, self.mpp, self.stream),
                   "gg_scale_pending")

    def asym_max(self, A, per_problem=False):
        n = self.lib.gg_sgl_nparts(self.p, self.M)
        out = torch.empty((self.M, n), dtype=torch.float64, device=self.dev)
        _lib.check(self.lib.gg_asym_max(_p(A), self.M, self.p, _p(out), self.stream), "gg_asym_max")
        if per_problem:
            return out.reshape(self.nprob, -1).amax(dim=1).cpu().numpy()
        return float(out.max().item())

    def is_posdef(self, A, res=None):
        """PD check of the reference (eigvalsh(Theta - L).min() > 0, admm_solver.py:294-296) without an extra
        eigendecomposition whenever a certificate is available:
          (1) Weyl: lambda_min(Theta-L) >= lambda_min(Omega) - |Omega-Theta+L|_F, with lambda_min(Omega) =
              phi+(min d) from the eigenvalues of the last Omega step (still resident) and the norm = the final
              primal residual r -- available for the non-latent 'boyd' loop;
          (2) a positive Gershgorin lower bound;
        otherwise the exact smallest eigenvalue is computed (min_eig)."""
        if self._weyl_certified(res):
            return True, None
        out = torch.empty(self.M, dtype=torch.float64, device=self.dev)
        _lib.check(self.lib.gg_gershgorin_min(_p(A), self.M, self.p, _p(self.eig.ws), self.eig.ws_bytes, _p(out),
                                              self.stream), "gg_gershgorin_min")
        if float(out.min().item()) > 0.0:
            return True, None
        d = self.min_eig(A)
        return d > 0, d

    def posdef_async(self, A, res=None):
        """like is_posdef, but when an eigendecomposition is needed it is only ENQUEUED (tridiagonal path: no host
        synchronisation) and a device scalar is returned, so the caller can overlap it with the D2H copies of the
        solution.  Returns None (certified PD) or a 0-d device tensor holding the smallest eigenvalue."""
        if self._weyl_certified(res):
            return None
        return self.eigvalsh(A).min()

    def _weyl_certified(self, res):
        """certificate (1) of is_posdef, from the loop's info ``res``: lambda_min(Omega) - r > 0"""
        if res is None or self.latent or not res.get("D_is_W") or self.nprob != 1:
            return False
        n = int(res["iters"][0])
        r, rho_used = res["hist"][0, n - 1, 0], res["hist"][0, n - 1, 4]
        beta = (self.nk if self.nk is not None else torch.ones(self.M, dtype=torch.float64, device=self.dev)) / rho_used
        dmin = self.eig.D.min(dim=1).values
        lam_min_omega = 0.5 * (torch.sqrt(dmin * dmin + 4 * beta) + dmin)
        return float(lam_min_omega.min().item()) - float(r) > 0.0

    def eigvalsh(self, A):
        """eigenvalues (M, p), unordered, of every matrix of the stack A; A is left intact (the eigensolver works on a
        copy).  Only enqueued; the result is the workspace's D, overwritten by the next decomposition."""
        return self.eig.eigh(A.clone(), ctrl=None, mpp=1, vectors=0, stream=self.stream)

    def min_eig_per_problem(self, A):
        """smallest eigenvalue of each problem's matrices in A, or -- where the Gershgorin bound of all of them is
        positive -- that bound (a certificate of positive definiteness, like is_posdef); device tensor (nprob,).
        The eigendecomposition of the stack is enqueued only when some problem is not certified."""
        g = torch.empty(self.M, dtype=torch.float64, device=self.dev)
        _lib.check(self.lib.gg_gershgorin_min(_p(A), self.M, self.p, _p(self.eig.ws), self.eig.ws_bytes, _p(g),
                                              self.stream), "gg_gershgorin_min")
        g = g.reshape(self.nprob, -1).amin(dim=1)
        if bool((g > 0.0).all().item()):
            return g
        D = self.eigvalsh(A)
        return torch.where(g > 0.0, g, D.reshape(self.nprob, -1).amin(dim=1))

    def mark(self):
        """event on the main stream: everything enqueued so far (the ADMM loop) -- used as the dependency of the
        overlapped D2H so that it does not wait for work enqueued later (the PD-check eigendecomposition)."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        return ev

    def to_host_overlapped(self, tensors, after=None):
        """D2H of the solution arrays on a side stream (copy engine) while the main stream keeps computing."""
        side = getattr(self, "_side", None)
        if side is None:
            side = self._side = torch.cuda.Stream(device=self.dev)
        if after is not None:
            side.wait_event(after)
        else:
            side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            out = to_host_many(tensors)
        return out

    def min_eig(self, A):
        """smallest eigenvalue over the stack (post-loop PD checks; reference uses eigvalsh)."""
        return float(self.eigvalsh(A).min().item())


def run_admm(kind, S, Omega_0, Theta_0, X_0, *, lambda1, lambda2=None, reg=None, lam_mat=None, rho=1.0,
             max_iter=1000, tol=1e-7, rtol=1e-4, stopping_criterion="boyd", update_rho=True, verbose=False,
             measure=False, latent=False, mu=None, nk=None, header=None, check_every=None, trace=None,
             check_symmetric=False, pvec=None, Mblk=None, print_rho=False, state=None, K=None):
    """Run the device ADMM loop.  ``kind``: 'mgl' (one problem of K matrices) or 'sgl' (M problems).

    ``K`` ('mgl' only): matrices per problem.  The stacks then hold M/K independent MGL problems (ADMM_MGL_batch),
    problem q owning matrices q*K .. q*K+K-1 and control block q; ``lambda1`` / ``lambda2`` may be arrays of one value
    per problem.  Default: one problem of all M matrices.

    ``pvec``: one true size p_q <= p per problem of a ragged batch whose problems are padded to p with decoupled unit
    diagonal entries (S = Omega = Theta = I, X = 0); the padding is left out of the residual norms.  'sgl' (block_SGL)
    or non-latent 'mgl' with the Boyd criterion (block_MGL, always on full matrices).

    ``state``: an AdmmState of the same shapes from an earlier call (lambda grids): its buffers and eigensolver
    workspace are reused.
    Returns (state, info) where info carries iteration counts, status and histories (numpy).
    """
    S3 = S if S.ndim == 3 else S[None]       # numpy arrays or device tensors
    M, p, _ = S3.shape
    mpp = (M if K is None else K) if kind == "mgl" else 1
    if kind == "mgl" and M // mpp > 1:
        if measure or stopping_criterion != "boyd":
            raise NotImplementedError("a batch of MGL problems supports stopping_criterion='boyd' without measure only")
        if mpp > K_TILE_MAX:
            raise NotImplementedError(f"a batch of MGL problems needs K <= {K_TILE_MAX} (tile-pair prox), got K = {mpp}")
    if kind == "mgl" and pvec is not None and (latent or measure or stopping_criterion != "boyd" or mpp > K_TILE_MAX):
        raise NotImplementedError(f"a ragged batch of MGL problems supports the non-latent loop with "
                                  f"stopping_criterion='boyd' without measure and K <= {K_TILE_MAX} only")
    lambdas = (lambda1, lambda2) if kind == "mgl" else None      # the MGL kernels read them from the control block
    if state is not None:
        st = state
        assert st.M == M and st.p == p and st.mpp == mpp and st.latent == latent and st.hist_cap >= max_iter
        st.reset(Omega_0.reshape(S3.shape), None if Theta_0 is None else Theta_0.reshape(S3.shape),
                 None if X_0 is None else X_0.reshape(S3.shape), rho, lambdas=lambdas)
        st.stream = torch.cuda.current_stream().cuda_stream
    else:
        st = AdmmState(S3, Omega_0.reshape(S3.shape), None if Theta_0 is None else Theta_0.reshape(S3.shape),
                       None if X_0 is None else X_0.reshape(S3.shape), mpp, rho, max_iter, latent, nk=nk, mu=mu,
                       lam_mat=lam_mat, pvec=pvec, lambdas=lambdas)
    lib, stream = st.lib, st.stream
    nprob = st.nprob
    regi = {"GGL": 0, "FGL": 1}.get(reg, -1)
    if check_symmetric:
        for A in (st.S, st.Omega, st.Theta, st.X):
            assert st.asym_max(A) <= 1e-5, "input X is not symmetric"

    if kind == "mgl":
        nt = lib.gg_mgl_ntile(p)
        nparts_fused = nt * nt
    else:
        nparts_fused = lib.gg_sgl_nparts(p, M)
    ragged_mgl = kind == "mgl" and st.pvec is not None
    nparts_dual = lib.gg_sgl_nparts(p, M) * mpp
    # K beyond the shared-memory layout of the fused tile-pair prox (K x 272 doubles per CTA): the row-band prox of the
    # K-sharded path takes over on one device (pack -> band prox -> unpack fused with the dual update)
    big_K = kind == "mgl" and mpp > K_TILE_MAX
    # scalar lambdas of the kernel arguments; the MGL kernels read each problem's lambdas from its control block
    if kind == "mgl":
        lam1_arg, lam2_arg = float(np.ravel(lambda1)[0]), float(np.ravel(lambda2)[0])
    # Non-latent MGL on the tridiagonal eigensolver path: the iterations keep only the UPPER triangles of Theta, X and W
    # current (every consumer inside the loop reads nothing else; half the elementwise HBM traffic) and the lower
    # triangles are filled once after the loop -- prox_p's mirroring (ggl_helper.py:198-205) done once.
    # A ragged batch stays on full matrices (its components are <= 160, where the upper-triangle path saves little).
    upper = (kind == "mgl" and not latent and not big_K and not ragged_mgl and stopping_criterion == "boyd"
             and not measure and not _DEBUG_KEEP_INPUT and st.eig.nb2 == 0 and p > lib.gg_jacobi_max()
             and _env_int("GG_UPPER", 1) != 0)
    nparts_upper = lib.gg_mgl_upper_nparts(p) if kind == "mgl" else 0
    if upper:
        nparts_fused = nparts_upper
    nparts = nparts_dual if (latent or big_K) else nparts_fused
    vband = tband = blk_nrm = None
    if big_K:
        vband = torch.empty(M * p * p, dtype=torch.float64, device=st.dev)
        tband = torch.zeros(M * p * p, dtype=torch.float64, device=st.dev)
    partials = torch.zeros((nprob, max(nparts_fused, nparts_dual, nparts_upper), NPART), dtype=torch.float64,
                           device=st.dev)
    if Mblk is not None:
        blk_nrm = torch.zeros((M, (p // Mblk) ** 2), dtype=torch.float64, device=st.dev)
    C = st.W if latent else None         # latent: the prox also forms C = Theta - X - Omega in W for the L step
    if check_every is None:
        check_every = 1 if (measure or verbose or p > 400) else 4
    runtime = np.zeros(max_iter)
    objective = np.zeros(max_iter)
    kkt_res = np.zeros(max_iter)
    obj_parts = None
    it_done = 0
    status = ""

    if verbose and header:
        print(header)
        if stopping_criterion == "boyd" and print_rho:
            print("%4s\t%10s\t%10s\t%10s\t%10s\t%10s" % ("iter", "r_t", "s_t", "eps_pri", "eps_dual", "rho"))
        elif stopping_criterion == "boyd":
            print("%4s\t%10s\t%10s\t%10s\t%10s" % ("iter", "r_t", "s_t", "eps_pri", "eps_dual"))
        else:
            print("%4s\t%10s" % ("iter", "kkt residual"))
    printed = 0

    for it in range(max_iter):
        if measure:
            torch.cuda.synchronize()
            t0 = time.time()
        st.omega_step(upper)
        if _DEBUG_KEEP_INPUT:
            _debug_check(st, it, "after omega_step", D=st.eig.D, Vt=st.W, Omega_new=st.Omega_new)
        if measure and kind == "mgl":
            # log det Omega_k = sum_i log phi+(d_i, beta_k) from the eigenvalues of W that are resident right now
            # (no extra eigendecomposition); tiny (K,p) reduction, kept on the device until the objective is formed
            beta = (st.nk if st.nk is not None else torch.ones(M, dtype=torch.float64, device=st.dev)) / st.ctrl[0, C_RHO]
            Dw = st.eig.D
            logdet_dev = torch.log(0.5 * (torch.sqrt(Dw * Dw + 4 * beta[:, None]) + Dw)).sum()
        Om, Om_prev, X, Th, ctl, parts = (_p(st.Omega_new), _p(st.Omega), _p(st.X), _p(st.Theta), _p(st.ctrl),
                                           _p(partials))
        if upper:
            _lib.check(lib.gg_prox_mgl_upper_batch(Om, Om_prev, X, Th, ctl, lam1_arg, lam2_arg, regi, mpp, p, nprob,
                                                   parts, stream), "gg_prox_mgl_upper")
        elif big_K:
            _lib.check(lib.gg_pack_bands(Om, _p(st.L), X, ctl, M, p, 1, _p(vband), stream), "gg_pack_bands")
            _lib.check(lib.gg_prox_band(_p(vband), _p(tband), ctl, lambda1, lambda2, regi, M, p, p, 0, stream),
                       "gg_prox_band")
            _lib.check(lib.gg_unpack_dual(_p(tband), Om, Om_prev, X, Th, _p(C), ctl, M, p, 1, parts, stream),
                       "gg_unpack_dual")
        elif ragged_mgl:
            _lib.check(lib.gg_prox_mgl_ragged(Om, Om_prev, X, Th, ctl, lam1_arg, lam2_arg, regi, mpp, p, nprob,
                                              _p(st.pvec), parts, stream), "gg_prox_mgl")
        elif kind == "mgl":
            _lib.check(lib.gg_prox_mgl_batch(Om, Om_prev, _p(st.L), X, Th, _p(C), ctl, lam1_arg, lam2_arg, regi, mpp,
                                             p, nprob, parts, stream), "gg_prox_mgl")
        elif Mblk is not None:
            _lib.check(lib.gg_prox_fsgl(Om, Om_prev, _p(st.L), X, Th, _p(C), ctl, float(lambda1), int(Mblk), M, p,
                                        parts, _p(blk_nrm), stream), "gg_prox_fsgl")
        else:
            _lib.check(lib.gg_prox_sgl(Om, Om_prev, _p(st.L), X, Th, _p(C), ctl, float(lambda1), _p(st.lam_mat), M, p,
                                       parts, _p(st.pvec), stream), "gg_prox_sgl")
        if _DEBUG_KEEP_INPUT:
            _debug_check(st, it, "after prox", Theta=st.Theta, X=st.X)
        if latent:
            st.l_step()
            _lib.check(lib.gg_dual_update(X, Om, Om_prev, Th, _p(st.L), ctl, M, p, mpp, 1 if kind == "sgl" else 0,
                                          parts, stream), "gg_dual_update")
        if measure:
            torch.cuda.synchronize()
            runtime[it] = time.time() - t0
            if kind == "mgl":
                objective[it] = _objective(st, st.Omega_new, lambda1, lambda2, regi, logdet_dev)
        it_done = it + 1
        if stopping_criterion == "boyd":
            _lib.check(lib.gg_stop_update(parts, nparts, ctl, _p(st.hist), st.hist_cap, _p(st.pdim), tol, rtol,
                                          1 if update_rho else 0, nprob, stream), "gg_stop_update")
            st.swap()
            # test hook: per-iteration state (X before the rho rescale, like the oracle); iterations after the done flag
            # are no-ops and are skipped
            if trace is not None and not (st.ctrl[0, C_DONE].item() != 0 and st.ctrl[0, C_ITER].item() != it + 1):
                if upper:
                    st.mirror()
                if callable(trace):
                    trace(st, it)
                else:
                    trace.append(dict(Omega=st.Omega.cpu().numpy(), Theta=st.Theta.cpu().numpy(),
                                      L=None if st.L is None else st.L.cpu().numpy(), X=st.X.cpu().numpy()))
            if (it + 1) % check_every == 0 or it + 1 == max_iter:
                ctrl = st.read_ctrl()
                if verbose and nprob == 1:
                    ndone = int(ctrl[0, C_ITER])
                    h = st.hist[0, printed:ndone].cpu().numpy()
                    for i, row in enumerate(h):
                        if print_rho:      # functional SGL prints the rho chosen for the NEXT iteration
                            rho_next = h[i + 1][4] if i + 1 < len(h) else ctrl[0, C_RHO]
                            print("%4d\t%10.4g\t%10.4g\t%10.4g\t%10.4g\t%10.4g" % (printed, row[0], row[1], row[2], row[3], rho_next))
                        else:
                            print("%4d\t%10.4g\t%10.4g\t%10.4g\t%10.4g" % (printed, row[0], row[1], row[2], row[3]))
                        printed += 1
                if np.all(ctrl[:, C_DONE] != 0):
                    break
        else:
            st.swap()
            eta = _kkt_residual(kind, st, lambda1, lambda2, regi, latent)
            kkt_res[it] = eta
            if verbose:
                print("%4d\t%10.4g" % (it, eta))
            if eta <= tol:
                status = "optimal"
                break

    st.finish_x()
    if upper:
        st.mirror()
    ctrl = st.read_ctrl()
    if stopping_criterion == "boyd" and np.any(ctrl[:, C_STATUS] < 0):
        bad = np.flatnonzero(ctrl[:, C_STATUS] < 0).tolist()
        raise _lib.GGLassoB200Error(f"non-finite residual in problem(s) {bad[:8]} after {int(ctrl[bad[0], C_ITER])} "
                                    "iteration(s): the input is not finite or an eigendecomposition broke down "
                                    "(numpy's eigh raises LinAlgError in the same situation)")
    info = {"ctrl": ctrl}
    if stopping_criterion == "boyd":
        iters = ctrl[:, C_ITER].astype(int)
        hist = st.hist.cpu().numpy()
        info["iters"] = iters
        info["hist"] = hist
        per_problem = [boyd_status(ctrl[q], hist[q]) for q in range(nprob)]
        info["status"] = [status for status, _ in per_problem]
        info["residual"] = [residual for _, residual in per_problem]
    else:
        info["iters"] = np.full(nprob, it_done)
        info["status"] = [status if status else "max iterations reached"] * nprob
        info["residual"] = [kkt_res[:it_done]] * nprob
    info["runtime"] = runtime
    info["objective"] = objective
    # st.eig.D still holds the eigenvalues of the last W (not overwritten by objective / KKT evaluations)
    info["D_is_W"] = (stopping_criterion == "boyd") and not latent
    return st, info


def _objective(st, Omega, lambda1, lambda2, regi, logdet):
    """f(Omega,S) + P(Theta) (admm_solver.py:213): <Omega,S> and P(Theta) from gg_objective, -log det from the
    eigenvalues of the Omega step (``logdet``: device scalar)."""
    lib = st.lib
    n = lib.gg_objective_nparts(st.p)
    parts = torch.empty((n, 2), dtype=torch.float64, device=st.dev)
    _lib.check(lib.gg_objective(_p(Omega), _p(st.S), _p(st.Theta), lambda1, lambda2, regi, st.M, st.p, _p(parts),
                                st.stream), "gg_objective")
    tot = parts.sum(0)
    return float((-logdet + tot[0] + tot[1]).item())


def _kkt_residual(kind, st, lambda1, lambda2, regi, latent):
    """KKT residual (admm_solver.py:333-371, single_admm_solver.py:293-319) from the device kernels.

    Elementwise glue (differences / norms of already-computed arrays) uses torch on the device;
    prox, eigendecomposition and spectral maps go through the same CUDA kernels as the loop.
    """
    lib, stream = st.lib, st.stream
    M, p = st.M, st.p
    ctrl1 = torch.from_numpy(control_block(st.nprob, 1.0)).to(st.dev, non_blocking=True)
    rho = st.ctrl[:, C_RHO].reshape(-1, 1, 1).repeat_interleave(st.mpp, 0)
    Xu = rho * st.X                                     # unscaled dual
    Omega, Theta = st.Omega, st.Theta
    L = st.L if latent else torch.zeros_like(Theta)
    zero = torch.zeros_like(Theta)
    P = torch.empty_like(Theta)
    Cdummy = torch.empty_like(Theta)
    if kind == "mgl" and M > K_TILE_MAX:
        _lib.check(lib.gg_add3(_p(Theta), _p(Xu), _p(zero), _p(Cdummy), M * p * p, stream), "gg_add3")
        _lib.check(lib.gg_prox_band(_p(Cdummy), _p(P), _p(ctrl1), lambda1, lambda2, regi, M, p, p, 0, stream),
                   "gg_prox_band")
    elif kind == "mgl":
        _lib.check(lib.gg_prox_mgl(_p(Theta), _p(Theta), _p(Xu), _p(zero), _p(P), _p(Cdummy), _p(ctrl1), lambda1,
                                   lambda2, regi, M, p, None, stream), "gg_prox_mgl")
    else:
        _lib.check(lib.gg_prox_sgl(_p(Theta), _p(Theta), _p(Xu), _p(zero), _p(P), _p(Cdummy), _p(ctrl1),
                                   float(lambda1), _p(st.lam_mat), M, p, None, None, stream), "gg_prox_sgl")
    nT = torch.linalg.norm(Theta)
    t1 = torch.linalg.norm(Theta - P) / (1 + nT)
    t2 = torch.linalg.norm(Theta - Omega - L) / (1 + nT)
    nk = st.nk.reshape(-1, 1, 1) if st.nk is not None else 1.0
    A = (Omega - nk * st.S - Xu).contiguous()
    st.eig.eigh(A, stream=stream)
    st.eig.recon(A, P, 0, bnum=st.nk, ctrl=None, stream=stream)
    t3 = torch.linalg.norm(Omega - P) / (1 + torch.linalg.norm(Omega))
    t4 = torch.zeros((), dtype=torch.float64, device=st.dev)
    if latent:
        A = (L - Xu).contiguous()
        st.eig.eigh(A, stream=stream)
        st.eig.recon(A, P, 1, bnum=st.mu, ctrl=None, stream=stream)
        t4 = torch.linalg.norm(L - P) / (1 + torch.linalg.norm(L))
    return float(torch.stack([t1, t2, t3, t4]).max().item())
