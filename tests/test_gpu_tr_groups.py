"""Stage 1 of the large-p eigensolver runs as concurrent chains over contiguous groups of the batch while the trailing
blocks are large (gg_tridiag.cu, gg_eigh_tridiag_impl), and as one chain over the batch otherwise.  Both kinds of
shape against LAPACK, problems marked done on either side of a group boundary, and four host threads solving at once.
"""
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

TR_TAIL = 144          # columns finished by the shared-memory tail kernel (gg_tridiag.cu)

SPLIT = [(20, 1000), (21, 1000), (2, 2047)]
NOT_SPLIT = [(3, 1000), (6, 384), (1, 1384)]


def _inputs(M, p, seed):
    """symmetric indefinite matrices with a diagonal and a rank-deficient member, as in test_eigh_matches_lapack"""
    rng = np.random.default_rng(seed)
    A = np.empty((M, p, p))
    for m in range(M):
        B = rng.standard_normal((p, p))
        A[m] = (B + B.T) / 2 - np.cov(rng.standard_normal((p, 2 * p + 2)), bias=True)
    A[0] = np.diag(np.arange(p, dtype=float))
    if M > 1:
        A[1][:, :2] = 0.0
        A[1][:2, :] = 0.0
    return A


def _check_lapack(A, D, Vt, ms=None):
    """eigenvalues, residual and orthogonality (eigenvectors as rows) with the tolerances of test_eigh_matches_lapack"""
    p = A.shape[1]
    ms = range(A.shape[0]) if ms is None else ms
    for m in ms:
        Dref = np.linalg.eigvalsh(A[m])
        scale = np.abs(Dref).max() + 1.0
        assert np.abs(np.sort(D[m]) - Dref).max() < 1e-11 * p ** 0.5 * scale, m
        Q = Vt[m].T
        assert np.abs(Q.T @ Q - np.eye(p)).max() < 1e-12, m
        assert np.abs(A[m] @ Q - Q * D[m]).max() < 2e-12 * p ** 0.5 * scale, m


def _eigh(A, ctrl=None, mpp=1, D_init=None, stream=None):
    from gglasso_b200._engine import Eigh, to_dev
    M, p = A.shape[:2]
    dev = torch.device("cuda")
    s = stream or torch.cuda.current_stream()
    with torch.cuda.stream(s):
        e = Eigh(M, p, dev)
        if D_init is not None:
            e.D.fill_(D_init)
        W = to_dev(A, dev)
        D = e.eigh(W, ctrl=ctrl, mpp=mpp, stream=s.cuda_stream)
        s.synchronize()
        return D.cpu().numpy(), W.cpu().numpy()


def _extra_launches(M, p):
    """launches of one tridiagonalisation beyond those of a single chain over the batch (zero: not split)"""
    from gglasso_b200 import _lib
    from gglasso_b200._engine import Eigh, _p
    lib = _lib.load()
    e = Eigh(M, p, torch.device("cuda"))
    W = torch.zeros((M, p, p), dtype=torch.float64, device="cuda")
    n0 = lib.gg_launch_count()
    _lib.check(lib.gg_sytrd_profile(_p(W), _p(e.D), M, p, _p(e.ws), e.ws_bytes, 0,
                                    torch.cuda.current_stream().cuda_stream), "gg_sytrd_profile")
    torch.cuda.synchronize()
    single = 4 + 2 * (p - TR_TAIL) + 1      # skip flags + 3 zero fills, column step + tile pass per column, tail
    return lib.gg_launch_count() - n0 - single


@pytest.mark.parametrize("M,p", SPLIT)
def test_split_shapes_match_lapack(M, p):
    assert _extra_launches(M, p) > 0
    A = _inputs(M, p, seed=M * 7919 + p)
    D, Vt = _eigh(A)
    _check_lapack(A, D, Vt)


@pytest.mark.parametrize("M,p", NOT_SPLIT)
def test_unsplit_shapes_match_lapack(M, p):
    assert _extra_launches(M, p) == 0
    A = _inputs(M, p, seed=M * 7919 + p)
    D, Vt = _eigh(A)
    _check_lapack(A, D, Vt)


def test_done_problems_across_the_group_boundary():
    """M = 21 splits 10 + 11; with three matrices per problem, problem 3 (matrices 9..11) straddles the boundary.
    Matrices of done problems come back untouched (input in A, D as it was), the others are solved."""
    from gglasso_b200 import _lib
    M, p, mpp = 21, 1000, 3
    assert _extra_launches(M, p) > 0
    A = _inputs(M, p, seed=5)
    ctrl = torch.zeros((M // mpp, _lib.CTRL_STRIDE), dtype=torch.float64, device="cuda")
    done = [0, 3]
    ctrl[done, _lib.C_DONE] = 1.0
    D, Vt = _eigh(A, ctrl=ctrl, mpp=mpp, D_init=-7.25)
    skipped = [m for m in range(M) if m // mpp in done]
    assert skipped == [0, 1, 2, 9, 10, 11]
    for m in skipped:
        assert np.array_equal(Vt[m], A[m]), m
        assert np.all(D[m] == -7.25), m
    _check_lapack(A, D, Vt, ms=[m for m in range(M) if m not in skipped])


def test_four_host_threads_match_single_thread():
    """four host threads, each on its own stream, solve at a split shape at the same time: every thread's result must
    equal the single-thread result for its input (up to the last-bit variation of the FP64 atomics)"""
    M, p, T = 10, 1000, 4
    assert _extra_launches(M, p) > 0
    inputs = [_inputs(M, p, seed=100 + t) for t in range(T)]
    single = [_eigh(A) for A in inputs]
    results, errors = [None] * T, []
    barrier = threading.Barrier(T)

    def work(t):
        try:
            torch.cuda.set_device(0)
            s = torch.cuda.Stream()
            barrier.wait()
            results[t] = _eigh(inputs[t], stream=s)
        except Exception as exc:       # reported below, on the main thread
            errors.append(exc)

    threads = [threading.Thread(target=work, args=(t,)) for t in range(T)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for t in range(T):
        D1, V1 = single[t]
        Dt, Vtt = results[t]
        scale = np.abs(D1).max() + 1.0
        assert np.abs(np.sort(Dt, 1) - np.sort(D1, 1)).max() < 1e-12 * p ** 0.5 * scale, t
        _check_lapack(inputs[t], Dt, Vtt)
