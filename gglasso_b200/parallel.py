"""Multi-GPU partitioning of the ADMM hot path (one process per GPU, torch.distributed).

Three natural seams (SURVEY.md section 8e):

* ``ADMM_MGL_dist``   one large-K MGL solve: the K instances are sharded across ranks for everything
                      that is per instance (W build, eigendecomposition, phi+ reconstruction, L step, dual
                      update); the cross-instance prox (``prox_p``, src/gglasso/solver/ggl_helper.py:190-207)
                      needs all K values of an entry, so ``V = Omega + L + X`` is re-tiled from instance layout
                      to row-band layout with one all-to-all, the prox runs on the band, and Theta travels
                      back with a second all-to-all.  The five residual sums are all-reduced (5 doubles) and
                      every rank takes the same rho / stopping decision.
* ``grid_search_dist`` lambda1 x lambda2 model-selection grid (src/gglasso/helper/model_selection.py:55-298):
                      lambda1 columns are dealt to ranks; inside a column the reference's warm-start chain
                      (``Omega_0 = previous Omega``, :224) is kept; no collective during the solves, one
                      gather of the per-grid-point scores at the end.
* ``assign_blocks``   LPT assignment of block_SGL's connected components (cost ~ size^3) to ranks.

The re-tile helpers work on CPU tensors over gloo as well, which is how the host logic is tested without GPUs.
"""
import os

import numpy as np
import torch
import torch.distributed as dist


def partition(n, parts):
    """balanced contiguous partition of range(n) into ``parts`` pieces -> list of (lo, hi)."""
    base, rem = divmod(n, parts)
    out, lo = [], 0
    for r in range(parts):
        hi = lo + base + (1 if r < rem else 0)
        out.append((lo, hi))
        lo = hi
    return out


def band_layout_index(K_loc, p, world):
    """index map of the all-to-all buffers written by gg_pack_bands / read by gg_unpack_dual: element (k, r, c) of
    this rank's (K_loc, p, p) stack sits at ``idx[k, r, c]`` of the flat buffer -- band d = partition(p, world)[d] of
    all local instances is one contiguous block [K_loc][rows_d][p].  Host-side statement of the CUDA layout (tests)."""
    idx = np.empty((K_loc, p, p), dtype=np.int64)
    col = np.arange(p)
    for lo, hi in partition(p, world):
        rows = hi - lo
        for k in range(K_loc):
            r = np.arange(lo, hi)
            idx[k, lo:hi, :] = K_loc * p * lo + ((k * rows + (r - lo)) * p)[:, None] + col[None, :]
    return idx


class KShard:
    """layout bookkeeping for a K-sharded (K_total, p, p) stack."""

    def __init__(self, K_total, p, group=None):
        # group=False forces a single-rank layout even inside an initialised process group
        local = group is False or not dist.is_initialized()
        self.group = None if local else group
        self.world = 1 if local else dist.get_world_size(group)
        self.rank = 0 if local else dist.get_rank(group)
        self.K_total, self.p = K_total, p
        self.kparts = partition(K_total, self.world)
        self.rparts = partition(p, self.world)
        self.k_lo, self.k_hi = self.kparts[self.rank]
        self.r_lo, self.r_hi = self.rparts[self.rank]
        self.K_loc = self.k_hi - self.k_lo
        self.nb = self.r_hi - self.r_lo

    # (K_loc, p, p) -> (K_total, nb, p): every rank ends up with its row band of ALL instances
    def to_band(self, x):
        p = self.p
        if self.world == 1:
            return x[:, self.r_lo:self.r_hi, :].contiguous()
        send = torch.cat([x[:, lo:hi, :].reshape(-1) for lo, hi in self.rparts])
        in_split = [self.K_loc * (hi - lo) * p for lo, hi in self.rparts]
        out_split = [(khi - klo) * self.nb * p for klo, khi in self.kparts]
        recv = torch.empty(sum(out_split), dtype=x.dtype, device=x.device)
        dist.all_to_all_single(recv, send, out_split, in_split, group=self.group)
        return recv.view(self.K_total, self.nb, p)

    # (K_total, nb, p) -> (K_loc, p, p)
    def from_band(self, y):
        p = self.p
        if self.world == 1:
            out = torch.empty((self.K_loc, p, p), dtype=y.dtype, device=y.device)
            out[:, self.r_lo:self.r_hi, :] = y
            return out
        y = y.contiguous()
        in_split = [(khi - klo) * self.nb * p for klo, khi in self.kparts]
        out_split = [self.K_loc * (hi - lo) * p for lo, hi in self.rparts]
        recv = torch.empty(sum(out_split), dtype=y.dtype, device=y.device)
        dist.all_to_all_single(recv, y.view(-1), out_split, in_split, group=self.group)
        out = torch.empty((self.K_loc, p, p), dtype=y.dtype, device=y.device)
        off = 0
        for (lo, hi), n in zip(self.rparts, out_split):
            out[:, lo:hi, :] = recv[off:off + n].view(self.K_loc, hi - lo, p)
            off += n
        return out

    def allreduce_sum(self, t):
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t


def ADMM_MGL_dist(S_local, lambda1, lambda2, reg, Omega_0_local, **kw):
    """K-sharded ADMM_MGL ('boyd' criterion).  Each rank passes ITS contiguous block of instances
    (rank r owns instances partition(K_total, world)[r]) and gets the matching block of the solution back.

    Keyword arguments: K_total, Theta_0_local, X_0_local, n_samples, tol, rtol, update_rho, rho, max_iter, verbose,
    latent, mu1_local, group, check_every.
    Returns (sol_local, info); info = {'status', 'iterations', 'residual'} identical on every rank.
    """
    from ._engine import to_host_many
    st, info = run_admm_mgl_dist(S_local, lambda1, lambda2, reg, Omega_0_local, **kw)
    latent = kw.get("latent", False)
    Omega = st.final_omega([info["iterations"]])
    outs = to_host_many([Omega, st.Theta, st.X] + ([st.L] if latent else []))
    sol = {"Omega": outs[0], "Theta": outs[1], "X": outs[2], "L": outs[3] if latent else np.zeros_like(S_local)}
    return sol, info


LAST_EXCHANGE = None        # how the last K-sharded solve exchanged its bands (diagnostics / tests)


class _P2PExchange:
    """receive buffers of the K-sharded loop in symmetric memory (torch.distributed._symmetric_memory): every rank
    allocates the same sizes (maxima over ranks), maps the peers' buffers and hands their device pointers to
    gg_pack_bands_p2p / gg_prox_band_p2p; `barrier` is the symmetric-memory barrier on the current stream."""

    def __init__(self, sh, dev):
        import ctypes
        import torch.distributed._symmetric_memory as symm
        group = sh.group if sh.group is not None else dist.group.WORLD
        p, world = sh.p, sh.world
        nb_max = max(hi - lo for lo, hi in sh.rparts)
        kl_max = max(hi - lo for lo, hi in sh.kparts)
        self.band_full = symm.empty(sh.K_total * nb_max * p, dtype=torch.float64, device=dev)
        self.back_full = symm.empty(kl_max * p * p, dtype=torch.float64, device=dev)
        self.hb = symm.rendezvous(self.band_full, group)
        self.hk = symm.rendezvous(self.back_full, group)
        self.band = self.band_full[:sh.K_total * sh.nb * p]
        self.back = self.back_full[:sh.K_loc * p * p]
        self.back.zero_()
        arr = ctypes.c_void_p * 16
        self.band_ptrs = arr(*[int(x) for x in self.hb.buffer_ptrs])
        self.back_ptrs = arr(*[int(x) for x in self.hk.buffer_ptrs])
        self.timeout_ms = int(os.environ.get("GG_DIST_P2P_TIMEOUT_MS", "20000"))

    def barrier(self, channel):
        self.hb.barrier(channel=channel, timeout_ms=self.timeout_ms)


_P2P_CACHE = {}


def _p2p_exchange(sh, dev):
    """None (with one warning) when symmetric memory cannot be set up on this machine: the NCCL all-to-all path runs.
    The buffers and the rendezvous are kept per (group, K_total, p): setting them up costs ~100 ms."""
    key = (id(sh.group), sh.K_total, sh.p, sh.world, dev.index)
    if key in _P2P_CACHE:
        return _P2P_CACHE[key]
    _P2P_CACHE[key] = ex = _p2p_exchange_new(sh, dev)
    return ex


def _p2p_exchange_new(sh, dev):
    try:
        ok = torch.tensor([1], dtype=torch.int32, device=dev)
        try:
            ex = _P2PExchange(sh, dev)
        except Exception as e:                          # noqa: BLE001  (any failure -> every rank must fall back)
            ex, ok[0] = None, 0
            import warnings
            warnings.warn(f"gglasso_b200: peer-memory exchange unavailable ({type(e).__name__}: {str(e)[:160]}); "
                          "using NCCL all-to-all")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=sh.group)
        if int(ok.item()) != 1:
            return None
        ex.barrier(2)                                   # every rank's buffers exist and are zeroed
        return ex
    except Exception:                                    # noqa: BLE001
        return None


def run_admm_mgl_dist(S_local, lambda1, lambda2, reg, Omega_0_local, K_total=None, Theta_0_local=None,
                      X_0_local=None, n_samples=None, tol=1e-5, rtol=1e-4, update_rho=True, rho=1., max_iter=1000,
                      verbose=False, latent=False, mu1_local=None, group=None, check_every=1):
    """device loop of ADMM_MGL_dist; returns (AdmmState, info) without copying the solution to the host."""
    from . import _lib
    from ._engine import AdmmState, _p, boyd_status
    from ._lib import C_DONE, C_ITER, C_STATUS, NPART
    assert reg in ['GGL', 'FGL'] and min(lambda1, lambda2) > 0 and rho > 0
    K_loc, p, _ = S_local.shape
    world = 1 if (group is False or not dist.is_initialized()) else dist.get_world_size(group)
    if K_total is None:
        t = torch.tensor([K_loc], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(t, group=group)
        K_total = int(t.item())
    sh = KShard(K_total, p, group)
    assert K_total >= sh.world, "K-sharded solve: every rank needs at least one instance (K_total >= world size)"
    assert sh.K_loc == K_loc, "each rank must hold partition(K_total, world)[rank] instances"
    nk = None if n_samples is None else np.asarray(n_samples, dtype=np.float64) * np.ones(K_loc)
    mu = None
    if latent:
        mu = (mu1_local * np.ones(K_loc)) if np.isscalar(mu1_local) else np.asarray(mu1_local, dtype=np.float64)
    st = AdmmState(S_local, Omega_0_local, Theta_0_local, X_0_local, K_loc, rho, max_iter, latent, nk=nk, mu=mu)
    st.pdim.fill_(K_total * ((p ** 2 + p) / 2))
    lib, stream = st.lib, st.stream
    regi = 0 if reg == "GGL" else 1
    nparts = lib.gg_sgl_nparts(p, K_loc) * K_loc
    partials = torch.zeros((nparts, NPART), dtype=torch.float64, device=st.dev)
    tot = torch.zeros((1, NPART), dtype=torch.float64, device=st.dev)
    # all-to-all buffers, allocated once: `send` = this rank's instances cut into row bands, `band` = this rank's row
    # band of ALL instances, `tband` = Theta on that band (kept across iterations: once the done flag is set the
    # kernels are no-ops and Theta stays what the last executed iteration produced), `back` = Theta of the local
    # instances, band by band.  With one rank the exchanges are the identity and the buffers alias.
    loc_n, band_n = K_loc * p * p, K_total * sh.nb * p
    p2p = _p2p_exchange(sh, st.dev) if (sh.world > 1 and os.environ.get("GG_DIST_P2P", "0") == "1") else None
    global LAST_EXCHANGE
    LAST_EXCHANGE = "single rank" if sh.world == 1 else ("peer memory" if p2p is not None else "nccl all-to-all")
    if p2p is None:
        send = torch.empty(loc_n, dtype=torch.float64, device=st.dev)
        band = torch.empty(band_n, dtype=torch.float64, device=st.dev) if sh.world > 1 else send
        tband = torch.zeros(band_n, dtype=torch.float64, device=st.dev)
        back = torch.empty(loc_n, dtype=torch.float64, device=st.dev) if sh.world > 1 else tband
    else:
        band, back = p2p.band, p2p.back
    loc_split = [K_loc * (hi - lo) * p for lo, hi in sh.rparts]
    band_split = [(khi - klo) * sh.nb * p for klo, khi in sh.kparts]

    for it in range(max_iter):
        st.omega_step()
        if p2p is not None:
            # the re-tile kernels store straight into the peers' buffers over NVLink; a barrier after each replaces
            # the all-to-all (DESIGN.md section 5).  Buffers are reused safely: a rank passes the second barrier only
            # when every rank has finished its prox (= has read its band), and the first one only after its own unpack.
            _lib.check(lib.gg_pack_bands_p2p(_p(st.Omega_new), _p(st.L), _p(st.X), _p(st.ctrl), K_loc, p, sh.world,
                                             sh.k_lo, p2p.band_ptrs, stream), "gg_pack_bands_p2p")
            p2p.barrier(0)
            _lib.check(lib.gg_prox_band_p2p(_p(band), p2p.back_ptrs, _p(st.ctrl), float(lambda1), float(lambda2), regi,
                                            K_total, sh.nb, p, sh.r_lo, sh.world, stream), "gg_prox_band_p2p")
            p2p.barrier(1)
        else:
            _lib.check(lib.gg_pack_bands(_p(st.Omega_new), _p(st.L), _p(st.X), _p(st.ctrl), K_loc, p, sh.world,
                                         _p(send), stream), "gg_pack_bands")
            if sh.world > 1:
                dist.all_to_all_single(band, send, band_split, loc_split, group=sh.group)
            _lib.check(lib.gg_prox_band(_p(band), _p(tband), _p(st.ctrl), float(lambda1), float(lambda2), regi, K_total,
                                        sh.nb, p, sh.r_lo, stream), "gg_prox_band")
            if sh.world > 1:
                dist.all_to_all_single(back, tband, loc_split, band_split, group=sh.group)
        # Theta back in instance layout, fused with the dual update and the residual sums (non-latent) or with
        # C = Theta - X - Omega for the L step (latent)
        _lib.check(lib.gg_unpack_dual(_p(back), _p(st.Omega_new), _p(st.Omega), _p(st.X), _p(st.Theta),
                                      _p(st.W) if latent else None, _p(st.ctrl), K_loc, p, sh.world, _p(partials),
                                      stream), "gg_unpack_dual")
        if latent:
            st.l_step()
            _lib.check(lib.gg_dual_update(_p(st.X), _p(st.Omega_new), _p(st.Omega), _p(st.Theta), _p(st.L),
                                          _p(st.ctrl), K_loc, p, K_loc, 0, _p(partials), stream), "gg_dual_update")
        torch.sum(partials, 0, keepdim=True, out=tot)
        sh.allreduce_sum(tot)
        _lib.check(lib.gg_stop_update(_p(tot), 1, _p(st.ctrl), _p(st.hist), st.hist_cap, _p(st.pdim), tol, rtol,
                                      1 if update_rho else 0, 1, stream), "gg_stop_update")
        st.swap()
        if (it + 1) % check_every == 0 or it + 1 == max_iter:
            ctrl = st.read_ctrl()
            if verbose and sh.rank == 0:
                n = int(ctrl[0, C_ITER])
                h = st.hist[0, n - 1].cpu().numpy()
                print("%4d\t%10.4g\t%10.4g\t%10.4g\t%10.4g" % (n - 1, h[0], h[1], h[2], h[3]))
            if ctrl[0, C_DONE] != 0:
                break
    st.finish_x()
    ctrl = st.read_ctrl()
    if ctrl[0, C_STATUS] < 0:
        raise _lib.GGLassoB200Error(f"non-finite residual after {int(ctrl[0, C_ITER])} iteration(s): the input is not "
                                    "finite or an eigendecomposition broke down")
    n = int(ctrl[0, C_ITER])
    status, residual = boyd_status(ctrl[0], st.hist[0, :n].cpu().numpy())
    info = {"status": status, "iterations": n, "residual": residual}
    return st, info


# ------------------------------------------------------------------------------------------------
# lambda grid sharding
# ------------------------------------------------------------------------------------------------
def ebic_mgl(S, Theta, N, gamma):
    """extended BIC summed over instances (reference: src/gglasso/helper/model_selection.py:841-869,
    robust_logdet :884-894: -inf when the smallest eigenvalue is <= 1e-12)."""
    K, p, _ = S.shape
    total = 0.0
    for k in range(K):
        w = np.linalg.eigvalsh(Theta[k])
        logdet = np.log(w).sum() if w.min() > 1e-12 else -np.inf
        E = (np.count_nonzero(Theta[k]) - p) / 2
        total += N[k] * (np.sum(S[k] * Theta[k]) - logdet) + E * (np.log(N[k]) + 4 * np.log(p) * gamma)
    return total


def grid_search_dist(solver, S, N, reg, l1, l2, gamma=0.1, tol=1e-7, rtol=1e-7, group=None, score=ebic_mgl,
                     solver_kwargs=None):
    """lambda1 x lambda2 grid for conforming MGL problems, lambda1 columns dealt round-robin to ranks.

    Mirrors the loop of the reference's ``grid_search`` (columns = lambda1 values run outermost, lambda2
    innermost, warm start ``Omega_0 <- previous Omega`` inside a column).  Across columns the reference chains
    the warm start as well; here every column starts from the identity, which changes iteration counts but
    not the optimum (strictly convex problem) -- SURVEY.md section 7 "grid sharding vs warm-start chain".

    Returns (scores (len(l2), len(l1)), best_index (g1, g2), best_sol) on every rank.
    """
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    K, p, _ = S.shape
    l1 = np.asarray(l1, dtype=float)
    l2 = np.asarray(l2, dtype=float)
    scores = np.full((len(l2), len(l1)), np.nan)
    iters = np.zeros((len(l2), len(l1)), dtype=int)
    best, best_score, best_ix = None, np.inf, None
    kw = dict(solver_kwargs or {})
    for g2 in range(rank, len(l1), world):
        Omega_0 = np.repeat(np.eye(p)[None], K, 0)
        for g1 in range(len(l2)):
            sol, info = solver(S, l1[g2], l2[g1], reg, Omega_0, tol=tol, rtol=rtol, **kw)
            Omega_0 = sol["Omega"].copy()
            sc = score(S, sol["Theta"], N, gamma)
            scores[g1, g2] = sc
            if sc < best_score:
                best_score, best_ix, best = sc, (g1, g2), {k: v.copy() for k, v in sol.items()}
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, (scores, best_score, best_ix), group=group)
        scores = np.full_like(scores, np.nan)
        owner, owner_score = 0, np.inf
        for r, (sc, bs, bix) in enumerate(gathered):
            m = ~np.isnan(sc)
            scores[m] = sc[m]
            if bs < owner_score:
                owner, owner_score, best_ix = r, bs, bix
        obj = [best if rank == owner else None]
        dist.broadcast_object_list(obj, src=owner, group=group)
        best = obj[0]
    return scores, best_ix, best


def _score_device(st, Omega_unused, N, gamma, method):
    """eBIC / AIC of the current Theta on the device (reference: src/gglasso/helper/model_selection.py:813-869,
    robust_logdet :884-894).  Eigenvalues come from the CUDA eigensolver (values only); the remaining terms are
    reductions over arrays that are already resident."""
    K, p = st.M, st.p
    Theta = st.Theta
    D = st.eigvalsh(Theta)          # (K,p)
    dmin = D.min(dim=1).values
    logdet = torch.where(dmin > 1e-12, torch.log(D.clamp_min(1e-300)).sum(1), torch.full_like(dmin, -float("inf")))
    inner = (st.S * Theta).sum((1, 2))
    E = (torch.count_nonzero(Theta.reshape(K, -1), dim=1).to(torch.float64) - p) / 2
    Nd = torch.as_tensor(np.asarray(N, dtype=np.float64), device=st.dev)
    pen = E * (torch.log(Nd) + 4 * np.log(p) * gamma) if method == "eBIC" else E
    return float((Nd * (inner - logdet) + pen).sum().item())


def grid_search_device(S, N, reg, l1, l2, method="eBIC", gamma=0.1, tol=1e-7, rtol=1e-7, latent=False, mu1=None,
                       group=None, n_streams=1):
    """lambda1 x lambda2 grid with everything resident on the GPU: S is uploaded once, each grid point runs the
    device ADMM loop, is scored on the device (eBIC/AIC) and hands its Omega to the next point of the column as
    warm start without touching the host; only the winning solution is copied back.  Columns (lambda1 values) are
    dealt round-robin to the ranks of ``group`` (one process per GPU); see grid_search_dist for the semantics.

    ``n_streams`` > 1 additionally runs that many columns concurrently on this GPU (one worker thread and CUDA
    stream each) -- worthwhile when a single solve cannot fill the device (p of a few hundred).

    Returns (scores (len(l2), len(l1)), iterations (same shape), best_index (g1, g2), best_sol) on every rank.
    """
    from ._engine import run_admm, to_host, require_cuda, to_dev
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    assert method in ("eBIC", "AIC") and reg in ("GGL", "FGL")
    K, p, _ = S.shape
    dev = require_cuda()
    S_dev = to_dev(S, dev)
    l1 = np.asarray(l1, dtype=float)
    l2 = np.asarray(l2, dtype=float)
    scores = np.full((len(l2), len(l1)), np.nan)
    iters = np.zeros((len(l2), len(l1)), dtype=int)
    eye = torch.eye(p, dtype=torch.float64, device=dev).repeat(K, 1, 1)
    best, best_score, best_ix = None, np.inf, None
    mu = None
    if latent:
        mu = mu1 * np.ones(K) if np.isscalar(mu1) else np.asarray(mu1, dtype=np.float64)
    my_cols = list(range(rank, len(l1), world))
    n_streams = max(1, min(int(n_streams), len(my_cols))) if my_cols else 1

    def run_columns(cols, out):
        """one worker = one CUDA stream: its columns run back to back, warm starts stay on the device"""
        b, b_score, b_ix = None, np.inf, None
        st = None                                 # one state per worker: buffers and workspace are reused
        for g2 in cols:
            Omega_0 = eye
            for g1 in range(len(l2)):
                st, res = run_admm("mgl", S_dev, Omega_0, None, None, lambda1=float(l1[g2]), lambda2=float(l2[g1]),
                                   reg=reg, tol=tol, rtol=rtol, latent=latent, mu=mu, state=st)
                n = int(res["iters"][0])
                Omega_0 = st.final_omega(res["iters"])
                sc = _score_device(st, Omega_0, N, gamma, method)
                scores[g1, g2], iters[g1, g2] = sc, n
                if sc < b_score:
                    b_score, b_ix = sc, (g1, g2)
                    b = {"Omega": Omega_0.clone(), "Theta": st.Theta.clone(), "X": st.X.clone(),
                         "L": st.L.clone() if latent else None}
        out.append((b_score, b_ix, b))

    results = []
    if n_streams == 1:
        run_columns(my_cols, results)
    else:
        # the grid points of different columns are independent and, at these sizes, latency bound: several
        # columns share the GPU from worker threads on their own streams (ctypes releases the GIL in the C calls)
        import threading
        torch.cuda.synchronize()
        errs = []

        def worker(cols):
            try:
                torch.cuda.set_device(dev)
                with torch.cuda.stream(torch.cuda.Stream(device=dev)):
                    run_columns(cols, results)
                    torch.cuda.current_stream().synchronize()
            except Exception as ex:                     # surface worker failures in the caller
                errs.append(ex)

        threads = [threading.Thread(target=worker, args=(my_cols[w::n_streams],)) for w in range(n_streams)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        if errs:
            raise errs[0]
    for b_score, b_ix, b in results:
        if b is not None and b_score < best_score:
            best_score, best_ix, best = b_score, b_ix, b
    if best is not None:
        best = {k: (to_host(v) if v is not None else np.zeros((K, p, p))) for k, v in best.items()}
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, (scores, iters, best_score, best_ix), group=group)
        scores = np.full_like(scores, np.nan)
        owner, owner_score = 0, np.inf
        for r, (sc, itr, bs, bix) in enumerate(gathered):
            m = ~np.isnan(sc)
            scores[m] = sc[m]
            iters[m] = itr[m]
            if bs < owner_score:
                owner, owner_score, best_ix = r, bs, bix
        obj = [best if rank == owner else None]
        dist.broadcast_object_list(obj, src=owner, group=group)
        best = obj[0]
    return scores, iters, best_ix, best


def block_SGL_dist(S, lambda1, Omega_0, Theta_0=None, X_0=None, rho=1., max_iter=1000, tol=1e-7, rtol=1e-3,
                   stopping_criterion="boyd", update_rho=True, lambda1_mask=None, group=None, solver=None):
    """block_SGL (src/gglasso/solver/single_admm_solver.py:326-475) with the connected components distributed over
    the ranks: every rank computes the same components and the same LPT assignment (cost ~ size^3), solves its
    share (small blocks as ragged batches on its GPU), and the disjoint block results are combined with one
    all-reduce(sum) per output array.  ``solver`` (default: the B200 ADMM_SGL) is injectable for CPU tests."""
    from .solver.single_admm_solver import _solve_components, get_connected_components
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    p = S.shape[0]
    mask = np.ones((p, p)) if lambda1_mask is None else lambda1_mask
    Theta_0 = Omega_0.copy() if Theta_0 is None else Theta_0
    X_0 = np.zeros((p, p)) if X_0 is None else X_0
    numC, allC = get_connected_components(S, lambda1 * mask)
    owner = assign_blocks([len(C) for C in allC], world)
    mine = [ci for ci in range(numC) if owner[ci] == rank]
    kw = dict(tol=tol, rtol=rtol, stopping_criterion=stopping_criterion, update_rho=update_rho, rho=rho,
              max_iter=max_iter, verbose=False, measure=False)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        sol = _solve_components(S, lambda1, mask, Omega_0, Theta_0, X_0, allC, mine, kw, solver=solver)
    if world > 1:
        # only the solved blocks travel (a few tens of MB at cfg5), not three dense p x p arrays: every rank sends the
        # diagonal blocks of its components and scatters what it receives; singletons were computed by their owners too
        mine_blocks = {ci: tuple(np.ascontiguousarray(sol[k][np.ix_(allC[ci], allC[ci])]) for k in ("Omega", "Theta", "X"))
                       for ci in mine}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine_blocks, group=group)
        for r, blocks in enumerate(gathered):
            if r == rank:
                continue
            for ci, (om, th, xx) in blocks.items():
                ix = np.ix_(allC[ci], allC[ci])
                sol["Omega"][ix], sol["Theta"][ix], sol["X"][ix] = om, th, xx
    return sol


def assign_blocks(sizes, world):
    """longest-processing-time assignment of connected components (cost ~ size^3) to ranks."""
    order = np.argsort(-np.asarray(sizes, dtype=float) ** 3, kind="stable")
    load = np.zeros(world)
    owner = np.zeros(len(sizes), dtype=int)
    for i in order:
        r = int(np.argmin(load))
        owner[i] = r
        load[r] += float(sizes[i]) ** 3
    return owner
