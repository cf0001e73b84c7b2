// gg_capi.cu -- extern "C" ABI (include/gglasso_b200.h) over the kernel launchers.
#include "../../include/gglasso_b200.h"
#include <cuda_runtime.h>
#include "gg_condat.cuh"

int gg_launch_build_w(const double*, const double*, double*, const double*, const double*, const double*, int, int,
                      int, double*, cudaStream_t);
int gg_launch_prox_sgl(const double*, const double*, const double*, double*, double*, double*, const double*, double,
                       const double*, int, int, double*, const int*, double*, int, cudaStream_t);
int gg_launch_dual_update(double*, const double*, const double*, const double*, const double*, const double*, int,
                          int, int, int, double*, cudaStream_t);
int gg_launch_prox_mgl(const double*, const double*, const double*, double*, double*, double*, const double*, double,
                       double, int, int, int, int, double*, cudaStream_t);
int gg_launch_prox_mgl_ragged(const double*, const double*, double*, double*, const double*, double, double, int, int,
                              int, int, const int*, double*, cudaStream_t);
int gg_launch_mgl_screen(const double*, const double*, double, double, int, int, int, uint32_t*, cudaStream_t);
int gg_launch_prox_mgl_upper(const double*, const double*, double*, double*, const double*, double, double, int, int,
                             int, int, double*, cudaStream_t);
int gg_launch_build_w_upper(const double*, double*, const double*, const double*, const double*, int, int, int,
                            double*, cudaStream_t);
int gg_launch_mirror_upper(double*, double*, int, int, cudaStream_t);
int gg_launch_stop_update(const double*, int, double*, double*, int, const double*, double, double, int, int,
                          cudaStream_t);
int gg_launch_scale_pending(double*, double*, int, int, int, cudaStream_t);
int gg_launch_objective(const double*, const double*, const double*, double, double, int, int, int, double*,
                        cudaStream_t);
int gg_launch_asym_max(const double*, int, int, double*, cudaStream_t);
int gg_launch_recon(const double*, const double*, const double*, const double*, int, int, int, int, double*,
                    cudaStream_t);
size_t gg_eigh_ws_bytes(int, int);
int gg_jacobi_small_max();
int gg_eigh_impl(double*, double*, int, int, const double*, int, void*, size_t, int, int, double, int, double, int*,
                 double*, cudaStream_t);

int gg_eigh_tridiag_impl(double*, double*, int, int, const double*, int, void*, size_t, cudaStream_t, int);
int gg_launch_add3(const double*, const double*, const double*, double*, size_t, cudaStream_t);
int gg_launch_ext_theta(const double*, const double*, const double*, const double*, const double*, const double*,
                        const double*, int, int, double*, double*, cudaStream_t);
int gg_launch_ext_lambda(const double*, const double*, const int*, int, int, int, double, const double*, double*,
                         cudaStream_t);
int gg_launch_ext_dual(double*, double*, const double*, const double*, const double*, const double*, const double*,
                       const double*, const double*, const int*, int, int, double*, cudaStream_t);
int gg_launch_prox_band(const double*, double*, const double*, double, double, int, int, int, int, int, cudaStream_t);
int gg_launch_pack_bands(const double*, const double*, const double*, const double*, int, int, int, double*, cudaStream_t);
int gg_launch_pack_bands_p2p(const double*, const double*, const double*, const double*, int, int, int, int, double* const*,
                             cudaStream_t);
int gg_launch_prox_band_p2p(const double*, double* const*, const double*, double, double, int, int, int, int, int, int,
                            cudaStream_t);
int gg_launch_unpack_dual(const double*, const double*, const double*, double*, double*, double*, const double*, int, int,
                          int, double*, cudaStream_t);
size_t gg_tridiag_ws_bytes(int, int);
int gg_sytrd_phase_times(unsigned long long*);
int gg_tr_lazy_depth();
int gg_gershgorin_min_impl(const double*, int, int, void*, size_t, double*, cudaStream_t);
int gg_launch_ppdna_build(const double*, const double*, const double*, const double*, const double*, double, double, int,
                          int, double*, double*, double*, const double*, cudaStream_t);
int gg_launch_ppdna_spectral(const double*, const double*, double, int, int, double*, double*, double*, double*,
                             const double*, cudaStream_t);
int gg_launch_ppdna_prox(const double*, const double*, const double*, const double*, const double*, const double*, double,
                         double, double, int, int, int, double*, double*, unsigned char*, double*, double*,
                         const double*, cudaStream_t);
int gg_launch_ppdna_jp(const double*, const double*, const unsigned char*, const double*, const double*, double, double,
                       int, int, int, double*, double*, const double*, cudaStream_t);
int gg_launch_ppdna_hess(const double*, const double*, const double*, const double*, const double*, const unsigned char*,
                         const double*, double, double, int, int, int, double*, double*, double*, double*,
                         const double*, cudaStream_t);
int gg_launch_ppdna_cg_init(const double*, int, int, double, int, double*, double*, double*, double*, double*,
                            cudaStream_t);
int gg_launch_ppdna_cg(int, const double*, const double*, const double*, const double*, const unsigned char*,
                       const double*, double, double, int, int, int, double*, double*, double*, double*, double*,
                       double*, double*, double*, cudaStream_t);
int gg_launch_subsample_cov(const double*, const int*, const int*, const int*, int, int, int, int, double*, double*, int*,
                            cudaStream_t);
int gg_launch_edge_count(const double*, int, int, int, int, int*, cudaStream_t);
int gg_launch_stars_instability(const int*, int, int, int, int, double*, cudaStream_t);

#include <atomic>
static std::atomic<long long> g_launches{0};
void gg_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

extern "C" {

long long gg_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int gg_sytrd_profile(double* A, double* D, int M, int p, void* ws, size_t ws_bytes, int which, void* stream)
{
    if (M <= 0 || p <= 32 || which < 0 || which > 2) return -1;
    if (ws_bytes < gg_tridiag_ws_bytes(M, p)) return -3;
    return gg_eigh_tridiag_impl(A, D, M, p, nullptr, 1, ws, ws_bytes, (cudaStream_t)stream, which == 0 ? 3 : which);
}

int gg_sytrd_write_depth(void) { return gg_tr_lazy_depth(); }

int gg_sytrd_phase_clock(unsigned long long* out16) { return gg_sytrd_phase_times(out16); }

int gg_jacobi_max(void) { return gg_jacobi_small_max(); }

int gg_version(void) { return 100; }

int gg_build_w(const double* Theta, const double* L, double* X, const double* S, const double* nk,
               const double* ctrl, int M, int p, int mpp, double* W, void* stream)
{
    if (M <= 0 || p <= 0 || mpp <= 0) return -1;
    return gg_launch_build_w(Theta, L, X, S, nk, ctrl, M, p, mpp, W, (cudaStream_t)stream);
}

size_t gg_eigh_workspace_bytes(int M, int p) { return gg_eigh_ws_bytes(M, p); }

int gg_eigh(double* A, double* D, int M, int p, const double* ctrl, int mpp, void* ws, size_t ws_bytes,
            int vectors, int block_nb2, double tol, int max_sweeps, double quad_tol, int* info, double* Vt_warm,
            void* stream)
{
    if (M < 0 || p < 0 || mpp <= 0) return -1;
    return gg_eigh_impl(A, D, M, p, ctrl, mpp, ws, ws_bytes, vectors, block_nb2, tol, max_sweeps, quad_tol, info,
                        Vt_warm, (cudaStream_t)stream);
}

int gg_recon(const double* Vt, const double* D, const double* bnum, const double* ctrl, int mpp, int mode, int M,
             int p, double* Out, void* stream)
{
    if (M <= 0 || p <= 0 || mpp <= 0 || mode < 0 || mode > 2) return -1;
    return gg_launch_recon(Vt, D, bnum, ctrl, mpp, mode, M, p, Out, (cudaStream_t)stream);
}

int gg_prox_sgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta, double* C,
                const double* ctrl, double lam, const double* lam_mat, int M, int p, double* partials, const int* pvec,
                void* stream)
{
    if (M <= 0 || p <= 0) return -1;
    return gg_launch_prox_sgl(Omega, Omega_prev, L, X, Theta, C, ctrl, lam, lam_mat, M, p, partials, pvec, nullptr, 0,
                              (cudaStream_t)stream);
}

int gg_prox_fsgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta, double* C,
                 const double* ctrl, double lam, int Mblk, int M, int p, double* partials, double* blk_nrm,
                 void* stream)
{
    if (M <= 0 || p <= 0 || Mblk <= 0 || p % Mblk != 0 || blk_nrm == nullptr) return -1;
    return gg_launch_prox_sgl(Omega, Omega_prev, L, X, Theta, C, ctrl, lam, nullptr, M, p, partials, nullptr, blk_nrm,
                              Mblk, (cudaStream_t)stream);
}

int gg_prox_mgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta, double* C,
                const double* ctrl, double lambda1, double lambda2, int reg, int K, int p, double* partials,
                void* stream)
{
    if (K <= 0 || p <= 0 || reg < 0 || reg > 1) return -1;
    return gg_launch_prox_mgl(Omega, Omega_prev, L, X, Theta, C, ctrl, lambda1, lambda2, reg, K, p, 1, partials,
                              (cudaStream_t)stream);
}

int gg_prox_mgl_batch(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                      double* C, const double* ctrl, double lambda1, double lambda2, int reg, int K, int p, int nprob,
                      double* partials, void* stream)
{
    if (K <= 0 || p <= 0 || nprob <= 0 || nprob > 65535 || reg < 0 || reg > 1 || ctrl == nullptr) return -1;
    return gg_launch_prox_mgl(Omega, Omega_prev, L, X, Theta, C, ctrl, lambda1, lambda2, reg, K, p, nprob, partials,
                              (cudaStream_t)stream);
}

int gg_prox_mgl_ragged(const double* Omega, const double* Omega_prev, double* X, double* Theta, const double* ctrl,
                       double lambda1, double lambda2, int reg, int K, int p, int nprob, const int* pvec,
                       double* partials, void* stream)
{
    if (K <= 0 || p <= 0 || nprob <= 0 || nprob > 65535 || reg < 0 || reg > 1 || ctrl == nullptr || pvec == nullptr
        || partials == nullptr)
        return -1;
    return gg_launch_prox_mgl_ragged(Omega, Omega_prev, X, Theta, ctrl, lambda1, lambda2, reg, K, p, nprob, pvec,
                                     partials, (cudaStream_t)stream);
}

int gg_mgl_screen(const double* S, const double* nk, double lambda1, double lambda2, int reg, int K, int p,
                  uint32_t* adj, void* stream)
{
    if (K <= 0 || p <= 0 || reg < 0 || reg > 1 || S == nullptr || adj == nullptr) return -1;
    return gg_launch_mgl_screen(S, nk, lambda1, lambda2, reg, K, p, adj, (cudaStream_t)stream);
}

int gg_prox_mgl_upper(const double* Omega, const double* Omega_prev, double* X, double* Theta, const double* ctrl,
                      double lambda1, double lambda2, int reg, int K, int p, double* partials, void* stream)
{
    if (K <= 0 || p <= 0 || reg < 0 || reg > 1) return -1;
    return gg_launch_prox_mgl_upper(Omega, Omega_prev, X, Theta, ctrl, lambda1, lambda2, reg, K, p, 1, partials,
                                    (cudaStream_t)stream);
}

int gg_prox_mgl_upper_batch(const double* Omega, const double* Omega_prev, double* X, double* Theta, const double* ctrl,
                            double lambda1, double lambda2, int reg, int K, int p, int nprob, double* partials,
                            void* stream)
{
    if (K <= 0 || p <= 0 || nprob <= 0 || nprob > 65535 || reg < 0 || reg > 1 || ctrl == nullptr) return -1;
    return gg_launch_prox_mgl_upper(Omega, Omega_prev, X, Theta, ctrl, lambda1, lambda2, reg, K, p, nprob, partials,
                                    (cudaStream_t)stream);
}

int gg_build_w_upper(const double* Theta, double* X, const double* S, const double* nk, const double* ctrl, int K,
                     int p, double* W, void* stream)
{
    if (K <= 0 || p <= 0) return -1;
    return gg_launch_build_w_upper(Theta, X, S, nk, ctrl, K, p, 1, W, (cudaStream_t)stream);
}

int gg_build_w_upper_batch(const double* Theta, double* X, const double* S, const double* nk, const double* ctrl, int K,
                           int p, int nprob, double* W, void* stream)
{
    if (K <= 0 || K > 65535 || p <= 0 || nprob <= 0 || nprob > 65535 || ctrl == nullptr) return -1;
    return gg_launch_build_w_upper(Theta, X, S, nk, ctrl, K, p, nprob, W, (cudaStream_t)stream);
}

int gg_mirror_upper(double* A0, double* A1, int M, int p, void* stream)
{
    if (M <= 0 || p <= 0 || A0 == nullptr) return -1;
    return gg_launch_mirror_upper(A0, A1, M, p, (cudaStream_t)stream);
}

int gg_dual_update(double* X, const double* Omega, const double* Omega_prev, const double* Theta, const double* L,
                   const double* ctrl, int M, int p, int mpp, int sgl_order, double* partials, void* stream)
{
    if (M <= 0 || p <= 0 || mpp <= 0) return -1;
    return gg_launch_dual_update(X, Omega, Omega_prev, Theta, L, ctrl, M, p, mpp, sgl_order, partials,
                                 (cudaStream_t)stream);
}

int gg_stop_update(const double* partials, int nparts, double* ctrl, double* hist, int hist_cap, const double* pdim,
                   double tol, double rtol, int update_rho, int nprob, void* stream)
{
    if (nparts <= 0 || nprob <= 0) return -1;
    return gg_launch_stop_update(partials, nparts, ctrl, hist, hist_cap, pdim, tol, rtol, update_rho, nprob,
                                 (cudaStream_t)stream);
}

int gg_scale_pending(double* X, double* ctrl, int M, int p, int mpp, void* stream)
{
    if (M <= 0 || p <= 0 || mpp <= 0) return -1;
    return gg_launch_scale_pending(X, ctrl, M, p, mpp, (cudaStream_t)stream);
}

int gg_objective(const double* Omega, const double* S, const double* Theta, double lambda1, double lambda2, int reg,
                 int K, int p, double* partials, void* stream)
{
    if (K <= 0 || p <= 0) return -1;
    return gg_launch_objective(Omega, S, Theta, lambda1, lambda2, reg, K, p, partials, (cudaStream_t)stream);
}

int gg_asym_max(const double* A, int M, int p, double* out, void* stream)
{
    if (M <= 0 || p <= 0) return -1;
    return gg_launch_asym_max(A, M, p, out, (cudaStream_t)stream);
}

int gg_add3(const double* Omega, const double* L, const double* X, double* V, size_t total, void* stream)
{
    if (total == 0) return 0;
    return gg_launch_add3(Omega, L, X, V, total, (cudaStream_t)stream);
}

int gg_prox_band(const double* V, double* Theta, const double* ctrl, double lambda1, double lambda2, int reg, int K,
                 int nb, int p, int row0, void* stream)
{
    if (K <= 0 || nb < 0 || p <= 0 || reg < 0 || reg > 1) return -1;
    return gg_launch_prox_band(V, Theta, ctrl, lambda1, lambda2, reg, K, nb, p, row0, (cudaStream_t)stream);
}

int gg_pack_bands(const double* Omega, const double* L, const double* X, const double* ctrl, int K_loc, int p, int world,
                  double* send, void* stream)
{
    if (K_loc <= 0 || p <= 0 || world <= 0 || world > p) return -1;
    return gg_launch_pack_bands(Omega, L, X, ctrl, K_loc, p, world, send, (cudaStream_t)stream);
}

int gg_pack_bands_p2p(const double* Omega, const double* L, const double* X, const double* ctrl, int K_loc, int p,
                      int world, int k_lo, double* const* peer_band, void* stream)
{
    if (K_loc <= 0 || p <= 0 || world <= 0 || world > 16 || world > p || k_lo < 0 || peer_band == nullptr) return -1;
    return gg_launch_pack_bands_p2p(Omega, L, X, ctrl, K_loc, p, world, k_lo, peer_band, (cudaStream_t)stream);
}

int gg_prox_band_p2p(const double* V, double* const* peer_back, const double* ctrl, double lambda1, double lambda2,
                     int reg, int K, int nb, int p, int row0, int world, void* stream)
{
    if (K <= 0 || nb < 0 || p <= 0 || reg < 0 || reg > 1 || world <= 0 || world > 16 || peer_back == nullptr) return -1;
    return gg_launch_prox_band_p2p(V, peer_back, ctrl, lambda1, lambda2, reg, K, nb, p, row0, world,
                                   (cudaStream_t)stream);
}

int gg_unpack_dual(const double* recv, const double* Omega, const double* Omega_prev, double* X, double* Theta,
                   double* C, const double* ctrl, int K_loc, int p, int world, double* partials, void* stream)
{
    if (K_loc <= 0 || p <= 0 || world <= 0 || world > p || ctrl == nullptr) return -1;
    return gg_launch_unpack_dual(recv, Omega, Omega_prev, X, Theta, C, ctrl, K_loc, p, world, partials,
                                 (cudaStream_t)stream);
}

int gg_ext_theta(const double* Omega, const double* L, const double* X0, const double* Lam, const double* X1,
                 const double* lam1, const double* ctrl, int K, int p, double* Theta, double* C, void* stream)
{
    if (K <= 0 || p <= 0) return -1;
    return gg_launch_ext_theta(Omega, L, X0, Lam, X1, lam1, ctrl, K, p, Theta, C, (cudaStream_t)stream);
}

int gg_ext_lambda(const double* Theta, const double* X1, const int* G, int Lg, int K, int p, double lambda2,
                  const double* ctrl, double* Lam, void* stream)
{
    if (K <= 0 || p <= 0 || Lg < 0) return -1;
    return gg_launch_ext_lambda(Theta, X1, G, Lg, K, p, lambda2, ctrl, Lam, (cudaStream_t)stream);
}

int gg_ext_dual(double* X0, double* X1, const double* Omega, const double* Omega_prev, const double* Theta,
                const double* L, const double* Lam, const double* Lam_prev, const double* ctrl, const int* pvec,
                int K, int p, double* partials, void* stream)
{
    if (K <= 0 || p <= 0) return -1;
    return gg_launch_ext_dual(X0, X1, Omega, Omega_prev, Theta, L, Lam, Lam_prev, ctrl, pvec, K, p, partials,
                              (cudaStream_t)stream);
}

int gg_gershgorin_min(const double* A, int M, int p, void* ws, size_t ws_bytes, double* out, void* stream)
{
    if (M <= 0 || p <= 0) return -1;
    return gg_gershgorin_min_impl(A, M, p, ws, ws_bytes, out, (cudaStream_t)stream);
}

void gg_host_tv1d(double* v, int n, int stride, double lam) { gg_tv1d_inplace(v, n, stride, lam); }

int gg_ppdna_build(const double* Omega_t, const double* Theta_t, const double* S, const double* X, const double* dX,
                   double s, double sigma, int K, int p, double* Xs, double* W, double* V, const double* flag,
                   void* stream)
{
    if (K <= 0 || p <= 0 || !(sigma > 0.0)) return -1;
    return gg_launch_ppdna_build(Omega_t, Theta_t, S, X, dX, s, sigma, K, p, Xs, W, V, flag, (cudaStream_t)stream);
}

int gg_ppdna_spectral(const double* Vt, const double* D, double sigma, int K, int p, double* Q, double* phi,
                      double* logdet, double* Omega, const double* flag, void* stream)
{
    if (K <= 0 || p <= 0 || !(sigma > 0.0)) return -1;
    return gg_launch_ppdna_spectral(Vt, D, sigma, K, p, Q, phi, logdet, Omega, flag, (cudaStream_t)stream);
}

int gg_ppdna_prox(const double* V, const double* Omega, const double* Omega_t, const double* Theta_t, const double* X,
                  const double* S, double lambda1, double lambda2, double sigma, int reg, int K, int p, double* Theta,
                  double* G, unsigned char* code, double* jscale, double* partials, const double* flag, void* stream)
{
    if (K <= 0 || p <= 0 || reg < 0 || reg > 1 || !(sigma > 0.0) || partials == nullptr) return -1;
    return gg_launch_ppdna_prox(V, Omega, Omega_t, Theta_t, X, S, lambda1, lambda2, sigma, reg, K, p, Theta, G, code,
                                jscale, partials, flag, (cudaStream_t)stream);
}

int gg_ppdna_jp(const double* Din, const double* V, const unsigned char* code, const double* jscale, const double* Jphi,
                double sigma, double lambda1, int reg, int K, int p, double* Out, double* partials, const double* flag,
                void* stream)
{
    if (K <= 0 || p <= 0 || reg < 0 || reg > 1) return -1;
    return gg_launch_ppdna_jp(Din, V, code, jscale, Jphi, sigma, lambda1, reg, K, p, Out, partials, flag,
                              (cudaStream_t)stream);
}

int gg_ppdna_hess(const double* Vt, const double* Q, const double* phi, const double* Din, const double* V,
                  const unsigned char* code, const double* jscale, double sigma, double lambda1, int reg, int K, int p,
                  double* Y, double* Z, double* Out, double* partials, const double* flag, void* stream)
{
    if (K <= 0 || p <= 0 || reg < 0 || reg > 1 || !(sigma > 0.0) || Out == Din) return -1;
    return gg_launch_ppdna_hess(Vt, Q, phi, Din, V, code, jscale, sigma, lambda1, reg, K, p, Y, Z, Out, partials, flag,
                                (cudaStream_t)stream);
}

int gg_ppdna_cg_init(const double* G, int K, int p, double tol, int max_iter, double* d, double* r, double* pv,
                     double* cg, double* partials, void* stream)
{
    if (K <= 0 || p <= 0) return -1;
    return gg_launch_ppdna_cg_init(G, K, p, tol, max_iter, d, r, pv, cg, partials, (cudaStream_t)stream);
}

int gg_ppdna_cg(int iters, const double* Vt, const double* Q, const double* phi, const double* V,
                const unsigned char* code, const double* jscale, double sigma, double lambda1, int reg, int K, int p,
                double* d, double* r, double* pv, double* q, double* Y, double* Z, double* cg, double* partials,
                void* stream)
{
    if (iters < 0 || K <= 0 || p <= 0 || reg < 0 || reg > 1 || !(sigma > 0.0)) return -1;
    return gg_launch_ppdna_cg(iters, Vt, Q, phi, V, code, jscale, sigma, lambda1, reg, K, p, d, r, pv, q, Y, Z, cg,
                              partials, (cudaStream_t)stream);
}

int gg_subsample_cov(const double* X, const int* rowoff, const int* idx, const int* boff, int nsub, int K, int p,
                     int scale, double* mean, double* S, int* zero_col, void* stream)
{
    if (nsub <= 0 || K <= 0 || p <= 0 || (long long)nsub * K > 65535 || !X || !rowoff || !idx || !boff || !mean || !S
        || !zero_col)
        return -1;
    return gg_launch_subsample_cov(X, rowoff, idx, boff, nsub, K, p, scale, mean, S, zero_col, (cudaStream_t)stream);
}

int gg_edge_count(const double* Theta, int nsub, int L, int K, int p, int* counts, void* stream)
{
    if (nsub <= 0 || L <= 0 || K <= 0 || p <= 0 || (long long)L * K > 65535 || !Theta || !counts) return -1;
    return gg_launch_edge_count(Theta, nsub, L, K, p, counts, (cudaStream_t)stream);
}

int gg_stars_instability(const int* counts, int L, int K, int p, int B, double* out, void* stream)
{
    if (L <= 0 || K <= 0 || p < 2 || B <= 0 || (long long)L * K > 2147483647LL || !counts || !out) return -1;
    return gg_launch_stars_instability(counts, L, K, p, B, out, (cudaStream_t)stream);
}

}  // extern "C"
