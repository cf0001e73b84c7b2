/*
 * gglasso_b200.h -- C ABI of the B200 (sm_100a) implementation of GGLasso's ADMM hot path.
 *
 * The reference (fabian-sp/GGLasso v0.2.1) is pure Python and has no FFI; its boundary for this
 * path is three Python callables (ADMM_MGL, ADMM_SGL, block_SGL).  The host side of this repo
 * (gglasso_b200/solver/) re-implements those callables and drives the entry points below through
 * ctypes.  Each entry point cites the reference code it replaces (paths relative to the
 * reference repository root).
 *
 * Conventions
 *   - all matrices are FP64, C-contiguous stacks (M, p, p) in DEVICE memory; M = number of
 *     matrices in the launch (K instances of one MGL problem, or M independent SGL problems);
 *   - `mpp` = matrices per ADMM problem (K for MGL, 1 for SGL batches); problem q = m / mpp;
 *   - `ctrl` = device control block, GG_CTRL_STRIDE doubles per problem (layout below); rho, the
 *     pending dual rescale and the done flag live there so the loop never needs the host;
 *   - `stream` is a cudaStream_t passed as void*;
 *   - return value: 0 on success, a positive cudaError_t, or a negative argument error;
 *   - no entry point allocates device memory: scratch comes from the caller
 *     (gg_eigh_workspace_bytes).
 */
#ifndef GGLASSO_B200_H
#define GGLASSO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GG_CTRL_STRIDE 16 /* doubles per problem */
/* ctrl[0]=rho  ctrl[1]=pending X scale  ctrl[2]=done  ctrl[3]=iterations done
 * ctrl[4..7]=r,s,eps_pri,eps_dual of the last iteration  ctrl[8]=1 if 'optimal'
 * ctrl[9], ctrl[10]: if ctrl[9] > 0, lambda1 / lambda2 of gg_prox_mgl and gg_prox_band are read from here instead of
 * the call arguments (lets a captured CUDA graph of one iteration serve every point of a lambda grid) */
#define GG_HIST_STRIDE 5  /* per iteration: r, s, eps_pri, eps_dual, rho */
#define GG_NPART 5        /* partial sums per CTA feeding gg_stop_update */

int gg_version(void);

/* number of kernels this library has launched in the calling process so far (monotonic; bench.py reports the
 * difference over its timed region as `gpu_launches`).  New; no reference counterpart. */
long long gg_launch_count(void);

/* W = Theta - L - X - (n_k/rho) S ; also folds the pending rescale of X (rho_old/rho_new) into X.
 * reference: src/gglasso/solver/admm_solver.py:180,236 ; single_admm_solver.py:163,205.
 * L may be NULL (non-latent); nk may be NULL (all ones) or a device array (M). */
int gg_build_w(const double* Theta, const double* L, double* X, const double* S, const double* nk,
               const double* ctrl, int M, int p, int mpp, double* W, void* stream);

/* Batched symmetric eigendecomposition (replaces np.linalg.eigh at admm_solver.py:181,199 and
 * single_admm_solver.py:164,174).  A (M,p,p) is overwritten by Vt: row c of Vt[m] is the unit
 * eigenvector belonging to D[m][c] (order and signs arbitrary).  vectors=0 skips normalisation
 * (eigenvalues only).  Path selection: p <= 48 shared-memory Jacobi (one CTA per matrix), larger p Householder
 * tridiagonalisation + divide & conquer + back-transformation.  block_nb2 = 0: default; 1: force the shared-memory
 * Jacobi kernel (p <= 160); 32/64/128: block-Jacobi with that many rows per block pair (p > 160).
 * tol<=0, max_sweeps<=0: defaults.  quad_tol: a sweep whose largest measured off-diagonal cosine is
 * below quad_tol is taken as the last one (quadratic convergence); 0 disables.  info[0] (host) = sweeps of the block
 * Jacobi, 0 for the shared-memory Jacobi (its sweep counts are not copied back), -1 for the tridiagonal path.
 * Vt_warm (optional, (M,p,p), rows orthonormal; used for p <= 160): warm start from the eigenvectors of the
 * previous ADMM iteration (identity for the first call); overwritten with the new eigenvectors. */
size_t gg_eigh_workspace_bytes(int M, int p);
int gg_eigh(double* A, double* D, int M, int p, const double* ctrl, int mpp, void* ws, size_t ws_bytes,
            int vectors, int block_nb2, double tol, int max_sweeps, double quad_tol, int* info, double* Vt_warm,
            void* stream);

/* Stage 1 of the large-p eigensolver only (Householder tridiagonalisation of the batch), for profiling:
 * which = 0 full sytrd, 1 only the per-column kernels, 2 only the trailing-matrix (symv + rank-2 update)
 * kernels.  Results of which != 0 are meaningless; A is destroyed.  p must exceed 32. */
int gg_sytrd_profile(double* A, double* D, int M, int p, void* ws, size_t ws_bytes, int which, void* stream);

/* Write-back depth q of the trailing-matrix kernel: pass j stores the updated trailing block only when q rank-2
 * updates are pending (every q-th pass moves 16 B per element, the others 8 B).  Needed to state the algorithmic
 * bytes of a launch; 1 <= q <= 4 (environment GG_TR_LAZY, default 3). */
int gg_sytrd_write_depth(void);
/* diagnostics (GG_TR_TIMING=1): nanoseconds per phase of the blocked tridiagonalisation's panel kernel, summed by one
 * CTA since the last call (16 counters, see gg_sytrd_blocked.cuh); reads and clears. */
int gg_sytrd_phase_clock(unsigned long long* out16);

/* Out = V diag(f(D)) V^T with V^T = Vt from gg_eigh (FP64 tensor cores, exactly symmetric result).
 * mode 0: f = phi+(d, beta) = (sqrt(d^2+4 beta)+d)/2   src/gglasso/solver/ggl_helper.py:272-303
 * mode 1: f = max(d-beta, 0)                            src/gglasso/solver/ggl_helper.py:29-36
 * mode 2: f = d
 * beta = bnum[m]/rho (bnum NULL -> 1; ctrl NULL -> rho = 1). */
int gg_recon(const double* Vt, const double* D, const double* bnum, const double* ctrl, int mpp, int mode,
             int M, int p, double* Out, void* stream);

/* Theta = prox_od_1norm(Omega + L + X, lam/rho)   src/gglasso/solver/ggl_helper.py:16-27,
 * single_admm_solver.py:169.  lam_mat (M,p,p) optional elementwise penalty (lambda1*lambda1_mask).
 * C == NULL (non-latent): fused with X += Omega - Theta (single_admm_solver.py:177) and the partial
 * sums for gg_stop_update (partials: M * gg_sgl_nparts(p,M) * GG_NPART doubles).
 * C != NULL (latent): writes C = Theta - X - Omega (single_admm_solver.py:173), X untouched.
 * pvec (optional, device int[M]): true size of problem m inside a padded (M,p,p) ragged batch (block_SGL's
 * connected components, single_admm_solver.py:441-459); entries beyond it are excluded from the norms. */
int gg_sgl_nparts(int p, int M);
int gg_prox_sgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                double* C, const double* ctrl, double lam, const double* lam_mat, int M, int p,
                double* partials, const int* pvec, void* stream);

/* Functional SGL: Theta = prox_sum_Frob(Omega + L + X, Mblk, lam/rho)   src/gglasso/solver/ggl_helper.py:45-66,
 * src/gglasso/solver/functional_sgl_admm.py:148.  Off-diagonal Mblk x Mblk blocks are shrunk in Frobenius norm.
 * blk_nrm: scratch, M * (p/Mblk)^2 doubles.  Same fusion / latent convention as gg_prox_sgl. */
int gg_prox_fsgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                 double* C, const double* ctrl, double lam, int Mblk, int M, int p, double* partials,
                 double* blk_nrm, void* stream);

/* Theta = prox_p(Omega + L + X, lambda1/rho, lambda2/rho, reg)   src/gglasso/solver/ggl_helper.py:190-207
 * reg 0 = GGL (ggl_helper.py:68-71,38-43), 1 = FGL (ggl_helper.py:131-134, fgl_helper.py:11-68).
 * Same fusion/latent convention as gg_prox_sgl; partials: gg_mgl_ntile(p)^2 * GG_NPART doubles,
 * zero-initialised by the caller once. */
int gg_mgl_ntile(int p);
int gg_prox_mgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                double* C, const double* ctrl, double lambda1, double lambda2, int reg, int K, int p,
                double* partials, void* stream);

/* The same prox + dual update + residual sums on the UPPER triangles only (non-latent loop; 2.5 A bytes instead of
 * 5 A): Theta and X are written for i <= j, the residual sums count off-diagonal entries twice.  The consumers inside
 * the loop (gg_build_w_upper, the tridiagonal path of gg_eigh) read upper triangles only; gg_mirror_upper fills the
 * lower triangles of up to two (M,p,p) stacks afterwards -- the mirroring of prox_p (ggl_helper.py:198-205) done once
 * instead of every iteration.  partials: gg_mgl_upper_nparts(p) * GG_NPART doubles.
 * gg_build_w_upper: W = Theta - X - (n_k/rho) S for i <= j (admm_solver.py:180), one problem of K instances. */
int gg_jacobi_max(void);   /* largest p solved by the shared-memory Jacobi kernel (which reads the full matrix) */
int gg_mgl_upper_nparts(int p);
int gg_prox_mgl_upper(const double* Omega, const double* Omega_prev, double* X, double* Theta, const double* ctrl,
                      double lambda1, double lambda2, int reg, int K, int p, double* partials, void* stream);
int gg_build_w_upper(const double* Theta, double* X, const double* S, const double* nk, const double* ctrl, int K,
                     int p, double* W, void* stream);
int gg_mirror_upper(double* A0, double* A1, int M, int p, void* stream);

/* Batches of nprob independent MGL problems of K instances each (ADMM_MGL_batch): the arrays are (nprob*K, p, p)
 * stacks, problem q owns matrices q*K .. q*K+K-1, control block q (done flag, rho, pending X scale and lambda1 /
 * lambda2 from ctrl[9..10], which must be set) and the partial sums at q * nparts * GG_NPART doubles, with nparts =
 * gg_mgl_ntile(p)^2 (gg_prox_mgl_batch) or gg_mgl_upper_nparts(p) (gg_prox_mgl_upper_batch) -- the layout
 * gg_stop_update reads for nprob problems.  Problems whose done flag is set are not touched.  Same kernels and
 * arithmetic as the single-problem entry points, which are the case nprob = 1; nprob <= 65535. */
int gg_prox_mgl_batch(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                      double* C, const double* ctrl, double lambda1, double lambda2, int reg, int K, int p, int nprob,
                      double* partials, void* stream);
int gg_prox_mgl_upper_batch(const double* Omega, const double* Omega_prev, double* X, double* Theta, const double* ctrl,
                            double lambda1, double lambda2, int reg, int K, int p, int nprob, double* partials,
                            void* stream);
int gg_build_w_upper_batch(const double* Theta, double* X, const double* S, const double* nk, const double* ctrl, int K,
                           int p, int nprob, double* W, void* stream);

/* Ragged batch of non-latent MGL problems (block_MGL): gg_prox_mgl_batch's layout, arithmetic and Theta / X, with
 * problem q a pvec[q] x pvec[q] problem padded to p (padding S = Omega = Theta = I, X = 0, a fixed point of the
 * iteration): entries with i >= pvec[q] or j >= pvec[q] are left out of the five partial sums. */
int gg_prox_mgl_ragged(const double* Omega, const double* Omega_prev, double* X, double* Theta, const double* ctrl,
                       double lambda1, double lambda2, int reg, int K, int p, int nprob, const int* pvec,
                       double* partials, void* stream);

/* Exact component screen of MGL (reg 0 = GGL, 1 = FGL; K <= 90): adj (p rows of ceil(p/32) uint32 words) gets bit b
 * of word w in row i set iff j = 32 w + b > i and prox_P(s_ij) != 0 with s_ij = (nk[k] S_k[i][j])_k (nk == NULL:
 * weights 1) and P the prox penalty at rho = 1 (same routines and expressions as gg_prox_mgl).  Every other bit
 * (diagonal, lower triangle, tail past p) is 0.  Deterministic. */
int gg_mgl_screen(const double* S, const double* nk, double lambda1, double lambda2, int reg, int K, int p,
                  uint32_t* adj, void* stream);

/* K-sharded MGL (one process per GPU, SURVEY.md section 8e): V = (Omega + L) + X on the local instances
 * (L may be NULL), and the cross-instance prox on a row band: V, Theta are (K, nb, p) slabs holding global rows
 * row0..row0+nb-1 of all K instances (after the all-to-all re-tile).  Same prox as gg_prox_mgl. */
int gg_add3(const double* Omega, const double* L, const double* X, double* V, size_t total, void* stream);
/* The two re-tile passes of the K-sharded solve, fused with their neighbours (no torch.cat / strided copies on the
 * hot path).  The p rows are cut into `world` contiguous bands (first p % world bands one row longer); band d of the
 * K_loc local instances is the contiguous block [K_loc][rows_d][p] at offset K_loc*p*lo_d of `send` / `recv`, i.e.
 * exactly the split layout of the two all-to-all exchanges.
 *   gg_pack_bands : send = (Omega + L) + X   (admm_solver.py:190 argument of prox_p), L may be NULL
 *   gg_unpack_dual: Theta (instance layout) from `recv`; C == NULL: X += Omega - Theta and the five residual partial
 *                   sums (admm_solver.py:208,316-331; partials (K_loc * gg_sgl_nparts(p,K_loc), 5));
 *                   C != NULL (latent): C = Theta - X - Omega (admm_solver.py:197), dual update follows the L step. */
int gg_pack_bands(const double* Omega, const double* L, const double* X, const double* ctrl, int K_loc, int p, int world,
                  double* send, void* stream);
int gg_unpack_dual(const double* recv, const double* Omega, const double* Omega_prev, double* X, double* Theta,
                   double* C, const double* ctrl, int K_loc, int p, int world, double* partials, void* stream);

/* Peer-memory variants of the two exchange steps (buffers in symmetric memory, peer_*[r] = device pointer of rank
 * r's buffer as mapped into this process, world <= 16): gg_pack_bands_p2p stores V = (Omega+L)+X of this rank's
 * instances (global indices k_lo ..) straight into every rank's band buffer (K_total, rows_d, p); gg_prox_band_p2p
 * runs the band prox and stores Theta of instance k into its owner's receive buffer (layout of gg_unpack_dual's
 * `recv`).  The caller places a cross-rank barrier after each.  Same arithmetic as gg_pack_bands / gg_prox_band. */
int gg_pack_bands_p2p(const double* Omega, const double* L, const double* X, const double* ctrl, int K_loc, int p,
                      int world, int k_lo, double* const* peer_band, void* stream);
int gg_prox_band_p2p(const double* V, double* const* peer_back, const double* ctrl, double lambda1, double lambda2,
                     int reg, int K, int nb, int p, int row0, int world, void* stream);
int gg_prox_band(const double* V, double* Theta, const double* ctrl, double lambda1, double lambda2, int reg,
                 int K, int nb, int p, int row0, void* stream);

/* ext_ADMM_MGL, non-conforming group graphical lasso (src/gglasso/solver/ext_admm_solver.py:191-273, :330-347,
 * :394-453).  The K matrices of size p_k are padded to (K,p,p); pvec[k] = p_k; one problem (ctrl block 0), rho fixed.
 *  gg_ext_theta : Theta = prox_od_1norm((Omega+L+X0+Lambda-X1)/2, lam1[k]/(2 rho)); C = Theta-X0-Omega if C != NULL
 *  gg_ext_lambda: Lambda = prox_2norm_G(Theta + X1, G, lambda2/rho); G is the reference's (2,Lg,K) int array
 *  gg_ext_dual  : X0 += Omega-Theta+L, X1 += Theta-Lambda, partial sums laid out for gg_stop_update (nparts =
 *                 K * gg_sgl_nparts(p,K)) */
int gg_ext_theta(const double* Omega, const double* L, const double* X0, const double* Lam, const double* X1,
                 const double* lam1, const double* ctrl, int K, int p, double* Theta, double* C, void* stream);
int gg_ext_lambda(const double* Theta, const double* X1, const int* G, int Lg, int K, int p, double lambda2,
                  const double* ctrl, double* Lam, void* stream);
int gg_ext_dual(double* X0, double* X1, const double* Omega, const double* Omega_prev, const double* Theta,
                const double* L, const double* Lam, const double* Lam_prev, const double* ctrl, const int* pvec,
                int K, int p, double* partials, void* stream);

/* X += Omega - Theta + L and partial sums (latent variants; L may be NULL for the K-sharded non-latent loop)   admm_solver.py:208, single_admm_solver.py:177.
 * sgl_order selects the association order of the reference's SGL expression. */
int gg_dual_update(double* X, const double* Omega, const double* Omega_prev, const double* Theta,
                   const double* L, const double* ctrl, int M, int p, int mpp, int sgl_order,
                   double* partials, void* stream);

/* Boyd residuals, stopping test and rho update on the device   admm_solver.py:216-246,316-331.
 * hist: nprob * hist_cap * GG_HIST_STRIDE doubles; pdim[q] = K(p^2+p)/2 of problem q. */
int gg_stop_update(const double* partials, int nparts, double* ctrl, double* hist, int hist_cap,
                   const double* pdim, double tol, double rtol, int update_rho, int nprob, void* stream);

/* apply the pending rescale to X after the loop (admm_solver.py:236) and clear it */
int gg_scale_pending(double* X, double* ctrl, int M, int p, int mpp, void* stream);

/* objective pieces for measure=True   ggl_helper.py:162-176,266-270 ; basic_linalg.py:20-33.
 * partials: 2 * gg_objective_nparts(p) doubles: {<Omega,S>, P(Theta)} per CTA.  reg -1 skips P. */
int gg_objective_nparts(int p);
int gg_objective(const double* Omega, const double* S, const double* Theta, double lambda1, double lambda2,
                 int reg, int K, int p, double* partials, void* stream);

/* max |A - A^T| partials (symmetry warnings, admm_solver.py:284-291); out: M * gg_sgl_nparts(p,M) doubles */
int gg_asym_max(const double* A, int M, int p, double* out, void* stream);

/* out[m] = min_i (a_ii - sum_{j!=i} |a_ij|): Gershgorin lower bound of the spectrum.  A positive bound proves
 * positive definiteness, letting the post-loop PD check (admm_solver.py:294-296) skip its eigendecomposition.
 * ws: at least the gg_eigh workspace of the same (M,p). */
int gg_gershgorin_min(const double* A, int M, int p, void* ws, size_t ws_bytes, double* out, void* stream);

/* PPDNA, the proximal point dual Newton method for GGL / FGL (src/gglasso/solver/ppdna_solver.py PPA_subproblem:65,
 * PPDNA:160; ggl_helper.py:74-159,218-249,323-437).  One problem of K instances (K <= 90); X is the UNSCALED dual;
 * flag (device double, may be NULL): every kernel is a no-op once *flag != 0.
 *  gg_ppdna_build   : Xs = X + s dX (dX may be NULL), W = Omega_t - sigma (S + Xs), V = Theta_t + sigma Xs, full
 *                     matrices (replaces the W / V assembly of PPA_subproblem, ppdna_solver.py:88-100)
 *  gg_ppdna_spectral: from gg_eigh's Vt and eigenvalues D of W: Q = Vt^T, phi = phi+(D, sigma) (K,p), logdet[k] =
 *                     sum log phi, Omega = Vt^T diag(phi) Vt   (phiplus, ggl_helper.py:272-303)
 *  gg_ppdna_prox    : Theta = prox_p(V, sigma lambda1, sigma lambda2) (same device routines as gg_prox_mgl), G =
 *                     Theta - Omega, the Jacobian data of prox_p (code: (K,p,p) bytes, jscale: (p,p) doubles) and
 *                     gg_ppdna_nparts(p) x 6 partial sums {<S,Omega>, P(Theta), <X,Omega-Theta>, |Omega-Omega_t|^2,
 *                     |Theta-Theta_t|^2, |G|^2}; the caller zeroes partials once (eval_jacobian_prox_p,
 *                     ggl_helper.py:218-252; Phi_t, :357)
 *  gg_ppdna_jp      : Out = sigma (Jphi + J_P(V)[Din]) (Jphi may be NULL or alias Out); partials (may be NULL):
 *                     gg_ppdna_jp_nparts(p) values of <Din, Out>   (jacobian_prox_phi_*, ggl_helper.py:74-159)
 *  gg_ppdna_hess    : Out = sigma (Q (Gamma o (Q^T Din Q)) Q^T + J_P(V)[Din]), Gamma_ab = phi_a phi_b/(phi_a phi_b +
 *                     sigma), on FP64 tensor cores; Y, Z: (K,p,p) scratch   (hessian_Y, ggl_helper.py:361-370)
 *  gg_ppdna_cg_init : d = 0, r = pv = -G, CG state cg (8 doubles) armed with tol and the iteration cap
 *  gg_ppdna_cg      : enqueues `iters` CG iterations on H d = -G (no-ops once cg[3] != 0); cg[0] = |r|^2, cg[4] =
 *                     iterations done   (cg_ppdna, ggl_helper.py:372-409).  partials: at least 1184 doubles. */
int gg_ppdna_build(const double* Omega_t, const double* Theta_t, const double* S, const double* X, const double* dX,
                   double s, double sigma, int K, int p, double* Xs, double* W, double* V, const double* flag,
                   void* stream);
int gg_ppdna_spectral(const double* Vt, const double* D, double sigma, int K, int p, double* Q, double* phi,
                      double* logdet, double* Omega, const double* flag, void* stream);
int gg_ppdna_nparts(int p);
int gg_ppdna_prox(const double* V, const double* Omega, const double* Omega_t, const double* Theta_t, const double* X,
                  const double* S, double lambda1, double lambda2, double sigma, int reg, int K, int p, double* Theta,
                  double* G, unsigned char* code, double* jscale, double* partials, const double* flag, void* stream);
int gg_ppdna_jp_nparts(int p);
int gg_ppdna_jp(const double* Din, const double* V, const unsigned char* code, const double* jscale, const double* Jphi,
                double sigma, double lambda1, int reg, int K, int p, double* Out, double* partials, const double* flag,
                void* stream);
int gg_ppdna_hess(const double* Vt, const double* Q, const double* phi, const double* Din, const double* V,
                  const unsigned char* code, const double* jscale, double sigma, double lambda1, int reg, int K, int p,
                  double* Y, double* Z, double* Out, double* partials, const double* flag, void* stream);
int gg_ppdna_cg_init(const double* G, int K, int p, double tol, int max_iter, double* d, double* r, double* pv,
                     double* cg, double* partials, void* stream);
int gg_ppdna_cg(int iters, const double* Vt, const double* Q, const double* phi, const double* V,
                const unsigned char* code, const double* jscale, double sigma, double lambda1, int reg, int K, int p,
                double* d, double* r, double* pv, double* q, double* Y, double* Z, double* cg, double* partials,
                void* stream);

/* Stability selection (StARS, Liu, Roeder & Wasserman 2010; no reference counterpart).  The samples of K classes are
 * one (sum n_k, p) FP64 array X, class k starting at row rowoff[k] (device int[K]).  A chunk of nsub subsamples is
 * given by idx (device int): subsample s draws the b_k = boff[k+1] - boff[k] rows idx[s*boff[K] + boff[k] ..] (indices
 * within class k) from class k; boff: device int[K+1], boff[0] = 0.
 *  gg_subsample_cov    : S[s*K+k] = (1/b_k) Xc^T Xc with Xc the drawn rows of class k centred on their mean
 *                        (np.cov(X_sub, rowvar=False, bias=True)), on FP64 tensor cores, exactly symmetric; scale != 0
 *                        then divides by sqrt(S_ii) sqrt(S_jj) (the reference's scale_array_by_diagonal,
 *                        src/gglasso/helper/basic_linalg.py).  S: (nsub*K, p, p); mean: nsub*K*p doubles of scratch;
 *                        zero_col[s*K+k] (int, nsub*K) = smallest column whose drawn values are all equal (zero
 *                        variance), or a value >= p if there is none.  nsub*K <= 65535.
 *  gg_edge_count       : counts[l,k,i,j] += #{s < nsub : Theta[(s*L+l)*K+k][i][j] != 0} for i < j; counts (L,K,p,p)
 *                        int32, zeroed by the caller once, entries i >= j untouched; deterministic (no atomics).
 *  gg_stars_instability: per (l,k) of counts after B subsamples, theta = count/B: out[(l*K+k)*2] = sum_{i<j}
 *                        2 theta (1 - theta) / C(p,2), out[(l*K+k)*2+1] = sum_{i<j} count / B; deterministic. */
int gg_subsample_cov(const double* X, const int* rowoff, const int* idx, const int* boff, int nsub, int K, int p,
                     int scale, double* mean, double* S, int* zero_col, void* stream);
int gg_edge_count(const double* Theta, int nsub, int L, int K, int p, int* counts, void* stream);
int gg_stars_instability(const int* counts, int L, int K, int p, int B, double* out, void* stream);

/* Host-side execution of the exact device TV-prox routine (unit tests without a GPU). */
void gg_host_tv1d(double* v, int n, int stride, double lam);

#ifdef __cplusplus
}
#endif
#endif
