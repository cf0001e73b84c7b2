// gg_elementwise.cu -- HBM-bound kernels of the ADMM iteration (sm_100a).
//
//   gg_build_w        W = Theta - L - X - (n_k/rho) S            admm_solver.py:180, single_admm_solver.py:163
//   gg_prox_sgl       Theta = prox_od_1norm(Omega+L+X, lam/rho)   single_admm_solver.py:169, ggl_helper.py:16-27
//                     fused with X += Omega - Theta and the five residual partial sums (non-latent)
//   gg_prox_mgl       Theta = prox_p(Omega+L+X, l1/rho, l2/rho)   admm_solver.py:190-194, ggl_helper.py:190-207
//                     GGL: ggl_helper.py:68-71,38-43; FGL: ggl_helper.py:131-134 + fgl_helper.py:11-68
//                     same fusion; one CTA per 16x16 tile pair (I<=J), all K instances, mirrored write
//   gg_prox_mgl_ragged  the same for a ragged batch (block_MGL): padding left out of the partial sums
//   gg_dual_update    X += Omega - Theta + L + partial sums (latent) admm_solver.py:208, single_admm_solver.py:177
//   gg_stop_update    Boyd residuals, stopping test, rho update    admm_solver.py:216-246,316-331
//   gg_scale          X *= pending rho_old/rho_new                 admm_solver.py:236
//
// Compiled with -fmad=false: these kernels are bandwidth bound and the unfused arithmetic
// keeps every expression bit-identical to the numpy/numba reference.
#include "gg_common.cuh"
#include "gg_condat.cuh"

#define EW_THREADS 256
#define EW_UNROLL 4

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(EW_THREADS)
build_w_kernel(const double* __restrict__ Theta, const double* __restrict__ L, double* __restrict__ X,
               const double* __restrict__ S, const double* __restrict__ nk, const double* __restrict__ ctrl,
               int mpp, size_t pp, double* __restrict__ W)
{
    const int m = blockIdx.y;
    const double* c = ctrl + (size_t)(m / mpp) * GG_CTRL_STRIDE;
    if (c[GG_C_DONE] != 0.0) return;
    const double rho = c[GG_C_RHO];
    const double xs = c[GG_C_XSCALE];
    const double beta = (nk ? nk[m] : 1.0) / rho;
    const size_t base = (size_t)m * pp;
    const size_t stride = (size_t)gridDim.x * EW_THREADS;
    const bool rescale = (xs != 1.0);
    for (size_t e0 = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e0 < pp; e0 += stride * EW_UNROLL) {
        double th[EW_UNROLL], x[EW_UNROLL], s[EW_UNROLL], l[EW_UNROLL];
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            const size_t e = e0 + u * stride;
            if (e < pp) {
                th[u] = Theta[base + e];
                x[u] = X[base + e];
                s[u] = S[base + e];
                l[u] = L ? L[base + e] : 0.0;
            }
        }
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            const size_t e = e0 + u * stride;
            if (e < pp) {
                const double xv = rescale ? xs * x[u] : x[u];
                double w = th[u];
                if (L) w = w - l[u];
                w = w - xv;
                w = w - beta * s[u];
                W[base + e] = w;
                if (rescale) X[base + e] = xv;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// SGL prox (+ fused dual update and residual partials when C == nullptr).
// lam: scalar lambda1, lam_mat: optional (M,p,p) elementwise penalty (lambda1 * mask).
__global__ void __launch_bounds__(EW_THREADS)
prox_sgl_kernel(const double* __restrict__ Omega, const double* __restrict__ Omega_prev,
                const double* __restrict__ L, double* __restrict__ X, double* __restrict__ Theta,
                double* __restrict__ C, const double* __restrict__ ctrl, double lam,
                const double* __restrict__ lam_mat, int p, double* __restrict__ partials,
                const int* __restrict__ pvec, const double* __restrict__ blk_nrm, int Mblk)
{
    __shared__ double scratch[GG_NPART * 32];
    const int m = blockIdx.y;
    const double* c = ctrl + (size_t)m * GG_CTRL_STRIDE;
    if (c[GG_C_DONE] != 0.0) return;
    const int pb = pvec ? pvec[m] : p;       // ragged batches: entries beyond pb are padding, excluded from norms
    const double inv_rho = 1.0 / c[GG_C_RHO];
    const size_t pp = (size_t)p * p;
    const size_t base = (size_t)m * pp;
    const size_t stride = (size_t)gridDim.x * EW_THREADS;
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (size_t e0 = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e0 < pp; e0 += stride * EW_UNROLL) {
        double vom[EW_UNROLL], vx[EW_UNROLL], vl[EW_UNROLL], vp[EW_UNROLL], vlam[EW_UNROLL];
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {               // all loads of the batch first (memory-level parallelism)
            const size_t e = e0 + u * stride;
            if (e < pp) {
                vom[u] = Omega[base + e];
                vx[u] = X[base + e];
                vl[u] = L ? L[base + e] : 0.0;
                vp[u] = C ? 0.0 : Omega_prev[base + e];
                vlam[u] = lam_mat ? lam_mat[base + e] : lam;
            }
        }
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            const size_t e = e0 + u * stride;
            if (e >= pp) continue;
            const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
            const double om = vom[u], x = vx[u], l = vl[u];
            double a = om;
            if (L) a = a + l;
            a = a + x;
            const double thr = inv_rho * vlam[u];
            double th;
            if (blk_nrm) {
                // functional SGL (prox_sum_Frob, ggl_helper.py:45-66): off-diagonal MxM blocks are shrunk in
                // Frobenius norm, v*(a-l)/a with a = max(|block|_F, l); diagonal blocks are kept
                const int bi = i / Mblk, bj = j / Mblk, nbk = p / Mblk;
                if (bi == bj) th = a;
                else {
                    const double nr = blk_nrm[(size_t)m * nbk * nbk + (size_t)(bi < bj ? bi : bj) * nbk + (bi < bj ? bj : bi)];
                    const double aa = nr > thr ? nr : thr;
                    th = (a * (aa - thr)) / aa;
                }
            } else {
                th = (i == j) ? a : gg_soft(a, thr);
            }
            Theta[base + e] = th;
            if (C) {
                C[base + e] = (th - x) - om;          // C_t = Theta_t - X_t - Omega_t
            } else {
                const double xn = (x + om) - th;      // X_t + Omega_t - Theta_t (+ L_t = 0)
                X[base + e] = xn;
                if (i < pb && j < pb) {
                    const double d1 = om - th, d2 = om - vp[u];
                    acc[0] += om * om; acc[1] += th * th; acc[2] += xn * xn; acc[3] += d1 * d1; acc[4] += d2 * d2;
                }
            }
        }
    }
    if (!C) {
        gg_block_sum<GG_NPART>(acc, scratch);
        if (threadIdx.x == 0) {
            double* out = partials + ((size_t)m * gridDim.x + blockIdx.x) * GG_NPART;
#pragma unroll
            for (int i = 0; i < GG_NPART; ++i) out[i] = acc[i];
        }
    }
}

// Frobenius norms of the strictly-upper MxM blocks of A = (Omega + L) + X  (functional SGL): one warp per block.
__global__ void __launch_bounds__(256)
fsgl_block_norm_kernel(const double* __restrict__ Omega, const double* __restrict__ L, const double* __restrict__ X,
                       const double* __restrict__ ctrl, int p, int Mblk, double* __restrict__ blk_nrm)
{
    const int m = blockIdx.y;
    if (ctrl[(size_t)m * GG_CTRL_STRIDE + GG_C_DONE] != 0.0) return;
    const int nbk = p / Mblk;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int pair = blockIdx.x * 8 + wid;
    if (pair >= nbk * nbk) return;
    const int bi = pair / nbk, bj = pair % nbk;
    if (bi >= bj) return;
    const size_t base = (size_t)m * p * p;
    double ss = 0.0;
    for (int e = lane; e < Mblk * Mblk; e += 32) {
        const int r = e / Mblk, c = e % Mblk;
        const size_t idx = base + (size_t)(bi * Mblk + r) * p + bj * Mblk + c;
        double a = Omega[idx];
        if (L) a = a + L[idx];
        a = a + X[idx];
        ss += a * a;
    }
    ss = gg_warp_sum(ss);
    if (lane == 0) blk_nrm[(size_t)m * nbk * nbk + (size_t)bi * nbk + bj] = sqrt(ss);
}

// ------------------------------------------------------------------------------------------
// Dual update for the latent variants:  X <- X + Omega - Theta + L, plus residual partials.
__global__ void __launch_bounds__(EW_THREADS)
dual_update_kernel(double* __restrict__ X, const double* __restrict__ Omega, const double* __restrict__ Omega_prev,
                   const double* __restrict__ Theta, const double* __restrict__ L, const double* __restrict__ ctrl,
                   int mpp, size_t pp, int sgl_order, double* __restrict__ partials)
{
    __shared__ double scratch[GG_NPART * 32];
    const int m = blockIdx.y;
    const double* c = ctrl + (size_t)(m / mpp) * GG_CTRL_STRIDE;
    if (c[GG_C_DONE] != 0.0) return;
    const size_t base = (size_t)m * pp;
    const size_t stride = (size_t)gridDim.x * EW_THREADS;
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (size_t e0 = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e0 < pp; e0 += stride * EW_UNROLL) {
        double vom[EW_UNROLL], vth[EW_UNROLL], vx[EW_UNROLL], vl[EW_UNROLL], vp[EW_UNROLL];
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            const size_t e = e0 + u * stride;
            if (e < pp) {
                vom[u] = Omega[base + e]; vth[u] = Theta[base + e]; vx[u] = X[base + e];
                vl[u] = L ? L[base + e] : 0.0; vp[u] = Omega_prev[base + e];
            }
        }
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            const size_t e = e0 + u * stride;
            if (e >= pp) continue;
            const double om = vom[u], th = vth[u], x = vx[u], l = vl[u];
            const double res = L ? ((om - th) + l) : (om - th);       // Omega - Theta + L
            const double xn = sgl_order ? (L ? (((x + om) - th) + l) : ((x + om) - th)) : (x + res);
            X[base + e] = xn;
            const double tl = th - l, d2 = om - vp[u];
            acc[0] += om * om; acc[1] += tl * tl; acc[2] += xn * xn; acc[3] += res * res; acc[4] += d2 * d2;
        }
    }
    gg_block_sum<GG_NPART>(acc, scratch);
    if (threadIdx.x == 0) {
        double* out = partials + ((size_t)m * gridDim.x + blockIdx.x) * GG_NPART;
#pragma unroll
        for (int i = 0; i < GG_NPART; ++i) out[i] = acc[i];
    }
}

// ------------------------------------------------------------------------------------------
// MGL prox: one CTA per 16x16 tile pair (I <= J); thread (tr,tc) owns entry (I*16+tr, J*16+tc)
// and runs the K-vector prox in shared memory (layout [k][tr*17+tc]: conflict-free for any
// per-thread k, which matters for the data-dependent TV scan).  The mirrored tile (J,I) is
// produced by reading the same shared values transposed, so global traffic is coalesced both
// ways and Theta is exactly symmetric, as in the reference (prox_p mirrors the upper triangle).
#define PT 16
#define PLD 17
#define PSLOT (PT * PLD)   // 272

// blockIdx.y read afresh at every use: the batched MGL kernels form the offset of problem q from it after the register-
// heavy K-vector prox instead of keeping a 64-bit offset live across it (which costs registers / spills at the kernels'
// launch bounds)
__device__ __forceinline__ size_t gg_batch_offset(int K, int p)
{
    unsigned q;
    asm volatile("mov.u32 %0, %%ctaid.y;" : "=r"(q));
    return (size_t)q * K * ((size_t)p * p);
}

// Body of the tile-pair prox kernels.  RAGGED: problem q of the batch is a p_q x p_q problem (p_q = pvec[q]) padded to
// p with decoupled unit diagonal entries; the padding is prox'd like any entry (it stays a fixed point) but is left out
// of the five partial sums, as prox_sgl_kernel does with its pvec.
template <int REG, bool LATENT, bool RAGGED>
__device__ __forceinline__ void
prox_mgl_body(const double* __restrict__ Omega, const double* __restrict__ Omega_prev,
              const double* __restrict__ L, double* __restrict__ X, double* __restrict__ Theta,
              double* __restrict__ C, const double* __restrict__ ctrl, double lambda1, double lambda2,
              int K, int p, double* __restrict__ partials, const int* __restrict__ pvec)
{
    extern __shared__ double ysm[];                 // K * PSLOT
    __shared__ double scratch[GG_NPART * 32];
    // Only tile pairs I <= J are launched, in super-tile order: blockIdx.x = 16 * (super-tile pair) + (a, b), so that
    // CTAs which are resident together cover 4 x 4 neighbouring tiles.  Each k-slice of a 16 x 16 tile is a set of
    // 128-byte row segments 8 MB apart; with neighbouring tiles in flight both the tile side and the mirror side
    // touch 512 contiguous bytes per matrix row, which keeps DRAM pages open (row-major order gave that to the tile
    // side only).
    const int nt = (p + PT - 1) / PT, nst = (nt + 3) >> 2;
    int sp = blockIdx.x >> 4, SI = 0;
    while (sp >= nst - SI) { sp -= nst - SI; ++SI; }
    const int SJ = SI + sp;
    const int I = 4 * SI + ((blockIdx.x >> 2) & 3), J = 4 * SJ + (blockIdx.x & 3);
    if (I > J || J >= nt) return;
    // problem q = blockIdx.y of a batch: control block q, matrices q*K.. (offset qo, folded into the element
    // index so that the array arguments stay kernel parameters) and nt*nt partial sums
    const double* cq = ctrl + (size_t)blockIdx.y * GG_CTRL_STRIDE;
    if (cq[GG_C_DONE] != 0.0) return;
    const double inv_rho = 1.0 / cq[GG_C_RHO];
    if (cq[GG_C_LAM1] > 0.0) { lambda1 = cq[GG_C_LAM1]; lambda2 = cq[GG_C_LAM2]; }
    const double l1 = inv_rho * lambda1, l2 = inv_rho * lambda2;
    const int tr = threadIdx.x / PT, tc = threadIdx.x % PT;
    const size_t pp = (size_t)p * p;
    const int i = I * PT + tr, j = J * PT + tc;
    const bool valid = (i < p) && (j < p);
    const bool upper = valid && (I < J || tr <= tc);
    const int slot = tr * PLD + tc;

    // ---- phase A: gather the K-vector of (Omega + L) + X, prox in place --------------------
    if (upper) {
        const size_t e = gg_batch_offset(K, p) + (size_t)i * p + j;
#pragma unroll 8
        for (int k = 0; k < K; ++k) {
            double v = Omega[k * pp + e];
            if (LATENT) v = v + L[k * pp + e];
            v = v + X[k * pp + e];
            ysm[k * PSLOT + slot] = v;
        }
        if (i != j) {
            double* y = ysm + slot;
            if (REG == 0) {            // GGL: group soft threshold of the l1-soft-thresholded vector
                double ss = 0.0;
                for (int k = 0; k < K; ++k) {
                    const double u = gg_soft(y[k * PSLOT], l1);
                    y[k * PSLOT] = u;
                    ss += u * u;
                }
                const double nrm = sqrt(ss);
                const double a = nrm > l2 ? nrm : l2;
                const double f = a - l2;
                for (int k = 0; k < K; ++k) y[k * PSLOT] = (y[k * PSLOT] * f) / a;
            } else {                   // FGL: TV prox across k, then l1 soft threshold
                gg_tv1d_inplace(y, K, PSLOT, l2);
                for (int k = 0; k < K; ++k) y[k * PSLOT] = gg_soft(y[k * PSLOT], l1);
            }
        }
    }
    __syncthreads();

    // ---- phase B: write Theta (+C or X and partial sums) for tile (I,J) and its mirror ------
    // Both sides are handled in the same k-loop so that six independent global loads are in flight per
    // iteration (the kernel is latency bound on these re-reads: ncu long-scoreboard 46 %).
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    {
        const size_t qo = gg_batch_offset(K, p);
        const int sl0 = (I < J || tr <= tc) ? slot : (tc * PLD + tr);
        const bool ok0 = valid;
        const size_t e0 = qo + (size_t)i * p + j;
        const int i1 = J * PT + tr, j1 = I * PT + tc;          // element of the mirror tile (J,I)
        const bool ok1 = (I < J) && (i1 < p) && (j1 < p);
        const size_t e1 = qo + (size_t)i1 * p + j1;
        const int sl1 = tc * PLD + tr;                         // = value of its transpose (j1, i1)
        bool in0 = true, in1 = true;                           // entries that count in the partial sums
        if (RAGGED) {
            const int pb = pvec[blockIdx.y];
            in0 = (i < pb) && (j < pb);
            in1 = (i1 < pb) && (j1 < pb);
        }
        if (ok0 || ok1) {
            const size_t ea = ok0 ? e0 : e1, eb = ok1 ? e1 : e0;   // keep addresses valid when one side is off
#pragma unroll (LATENT ? 4 : 2)
            for (int k = 0; k < K; ++k) {
                const size_t o = (size_t)k * pp;
                const double om0 = Omega[o + ea], x0 = X[o + ea];
                const double om1 = Omega[o + eb], x1 = X[o + eb];
                double p0 = 0.0, p1 = 0.0;
                if (!LATENT) { p0 = Omega_prev[o + ea]; p1 = Omega_prev[o + eb]; }
                const double th0 = ysm[k * PSLOT + sl0], th1 = ysm[k * PSLOT + sl1];
                if (ok0) {
                    Theta[o + e0] = th0;
                    if (LATENT) {
                        C[o + e0] = (th0 - x0) - om0;
                    } else {
                        const double d1 = om0 - th0;
                        const double xn = x0 + d1;             // X += Omega - Theta (+ L = 0)
                        X[o + e0] = xn;
                        const double d2 = om0 - p0;
                        if (!RAGGED || in0) {
                            acc[0] += om0 * om0; acc[1] += th0 * th0; acc[2] += xn * xn; acc[3] += d1 * d1; acc[4] += d2 * d2;
                        }
                    }
                }
                if (ok1) {
                    Theta[o + e1] = th1;
                    if (LATENT) {
                        C[o + e1] = (th1 - x1) - om1;
                    } else {
                        const double d1 = om1 - th1;
                        const double xn = x1 + d1;
                        X[o + e1] = xn;
                        const double d2 = om1 - p1;
                        if (!RAGGED || in1) {
                            acc[0] += om1 * om1; acc[1] += th1 * th1; acc[2] += xn * xn; acc[3] += d1 * d1; acc[4] += d2 * d2;
                        }
                    }
                }
            }
        }
    }
    if (!LATENT) {
        gg_block_sum<GG_NPART>(acc, scratch);
        if (threadIdx.x == 0) {
            double* out = partials + (((size_t)blockIdx.y * nt + I) * nt + J) * GG_NPART;
#pragma unroll
            for (int q = 0; q < GG_NPART; ++q) out[q] = acc[q];
        }
    }
}

template <int REG, bool LATENT>
__global__ void __launch_bounds__(PT * PT)
prox_mgl_kernel(const double* __restrict__ Omega, const double* __restrict__ Omega_prev,
                const double* __restrict__ L, double* __restrict__ X, double* __restrict__ Theta,
                double* __restrict__ C, const double* __restrict__ ctrl, double lambda1, double lambda2,
                int K, int p, double* __restrict__ partials)
{
    prox_mgl_body<REG, LATENT, false>(Omega, Omega_prev, L, X, Theta, C, ctrl, lambda1, lambda2, K, p, partials,
                                      nullptr);
}

// ragged batch of non-latent problems (block_MGL): pvec[q] = true size of problem q
template <int REG>
__global__ void __launch_bounds__(PT * PT)
prox_mgl_ragged_kernel(const double* __restrict__ Omega, const double* __restrict__ Omega_prev,
                       double* __restrict__ X, double* __restrict__ Theta, const double* __restrict__ ctrl,
                       double lambda1, double lambda2, int K, int p, const int* __restrict__ pvec,
                       double* __restrict__ partials)
{
    prox_mgl_body<REG, false, true>(Omega, Omega_prev, nullptr, X, Theta, nullptr, ctrl, lambda1, lambda2, K, p,
                                    partials, pvec);
}

// ------------------------------------------------------------------------------------------
// W build on the upper triangle only (companion of prox_mgl_upper_kernel; non-latent MGL).  Rows i and p-1-i are
// handled by the same CTA (p+1 entries together), columns start at the 256-byte boundary left of the diagonal.
__global__ void __launch_bounds__(EW_THREADS)
build_w_upper_kernel(const double* __restrict__ Theta, double* __restrict__ X, const double* __restrict__ S,
                     const double* __restrict__ nk, const double* __restrict__ ctrl, int p, double* __restrict__ W)
{
    // matrix k = blockIdx.y of problem q = blockIdx.z (K = gridDim.y matrices per problem)
    const int m = blockIdx.z * gridDim.y + blockIdx.y;
    ctrl += (size_t)blockIdx.z * GG_CTRL_STRIDE;
    if (ctrl[GG_C_DONE] != 0.0) return;
    const double rho = ctrl[GG_C_RHO];
    const double xs = ctrl[GG_C_XSCALE];
    const double beta = (nk ? nk[m] : 1.0) / rho;
    const bool rescale = (xs != 1.0);
    const size_t base = (size_t)m * p * p;
    const int half = (p + 1) / 2;
    for (int r = blockIdx.x; r < half; r += gridDim.x) {
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const int i = side ? p - 1 - r : r;
            if (side && i == r) break;
            const size_t row = base + (size_t)i * p;
            for (int j = (i & ~31) + threadIdx.x; j < p; j += EW_THREADS) {
                if (j < i) continue;
                const double x = X[row + j];
                const double xv = rescale ? xs * x : x;
                double w = Theta[row + j];
                w = w - xv;
                w = w - beta * S[row + j];
                W[row + j] = w;
                if (rescale) X[row + j] = xv;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// MGL prox on the UPPER triangle only (non-latent loop).  Every array of the iteration is symmetric, and the kernels
// that consume Theta and X inside the loop need their upper triangles only: build_w forms W entry by entry and the
// tridiagonal eigensolver reads the upper triangle of W; the residual norms are sums in which an off-diagonal entry
// counts twice.  So the loop keeps the upper triangles of Theta and X current (2.5 A bytes instead of 5 A) and
// mirror_upper_kernel fills the lower ones once, after the last iteration -- the same mirroring prox_p does
// (ggl_helper.py:190-207), done once instead of every iteration.
// One CTA per tile of UT_R rows x UT_C columns: a warp reads 256 contiguous bytes per k-slice, a CTA row 256 B; CTAs
// that are resident together continue the same rows.  Thread t owns one entry; its K-vector lives in shared memory at
// [k][t] (distinct banks for any per-thread k, which the data-dependent TV scan needs).
#define UT_R 8
#define UT_C 32
#define UT_THREADS (UT_R * UT_C)

__host__ __device__ inline int ut_ntiles(int p)
{
    const int nr = (p + UT_R - 1) / UT_R, nc = (p + UT_C - 1) / UT_C;
    int n = 0;
    for (int I = 0; I < nr; ++I) n += nc - (I * UT_R) / UT_C;
    return n;
}

template <int REG>
__global__ void __launch_bounds__(UT_THREADS, 4)
prox_mgl_upper_kernel(const double* __restrict__ Omega, const double* __restrict__ Omega_prev,
                      double* __restrict__ X, double* __restrict__ Theta, const double* __restrict__ ctrl,
                      double lambda1, double lambda2, int K, int p, double* __restrict__ partials)
{
    extern __shared__ double ysm[];                 // K * UT_THREADS
    __shared__ double scratch[GG_NPART * 32];
    // problem q = blockIdx.y of a batch: control block q, matrices q*K.. (offset folded into the element index) and
    // gridDim.x partial sums
    const double* cq = ctrl + (size_t)blockIdx.y * GG_CTRL_STRIDE;
    if (cq[GG_C_DONE] != 0.0) return;
    // tile rows are grouped by UT_C / UT_R = 4: the rows of group g start at tile column g
    const int nc = (p + UT_C - 1) / UT_C;
    constexpr int GR = UT_C / UT_R;
    int rem = blockIdx.x, g = 0;
    while (rem >= GR * (nc - g)) { rem -= GR * (nc - g); ++g; }
    const int I = g * GR + rem / (nc - g), J = g + rem % (nc - g);
    const double inv_rho = 1.0 / cq[GG_C_RHO];
    if (cq[GG_C_LAM1] > 0.0) { lambda1 = cq[GG_C_LAM1]; lambda2 = cq[GG_C_LAM2]; }
    const double l1 = inv_rho * lambda1, l2 = inv_rho * lambda2;
    const int i = I * UT_R + threadIdx.x / UT_C, j = J * UT_C + threadIdx.x % UT_C;
    const size_t pp = (size_t)p * p;
    const bool own = (i < p) && (j < p) && (i <= j);
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (own) {
        double* y = ysm + threadIdx.x;
        {
            const size_t e = (size_t)i * p + j;
            const size_t qo = gg_batch_offset(K, p);
#pragma unroll 8
            for (int k = 0; k < K; ++k) y[k * UT_THREADS] = Omega[qo + k * pp + e] + X[qo + k * pp + e];
        }
        if (i != j) {
            if (REG == 0) {            // GGL: group soft threshold of the l1-soft-thresholded vector
                double ss = 0.0;
                for (int k = 0; k < K; ++k) {
                    const double u = gg_soft(y[k * UT_THREADS], l1);
                    y[k * UT_THREADS] = u;
                    ss += u * u;
                }
                const double nrm = sqrt(ss);
                const double a = nrm > l2 ? nrm : l2;
                const double f = a - l2;
                for (int k = 0; k < K; ++k) y[k * UT_THREADS] = (y[k * UT_THREADS] * f) / a;
            } else {                   // FGL: TV prox across k, then l1 soft threshold
                gg_tv1d_inplace(y, K, UT_THREADS, l2);
                for (int k = 0; k < K; ++k) y[k * UT_THREADS] = gg_soft(y[k * UT_THREADS], l1);
            }
        }
        const double w = (i == j) ? 1.0 : 2.0;      // an off-diagonal entry stands for itself and its mirror image
        const size_t e = (size_t)i * p + j;
#pragma unroll 4
        for (int k = 0; k < K; ++k) {
            const size_t o = gg_batch_offset(K, p) + (size_t)k * pp + e;
            const double om = Omega[o], x = X[o], pv = Omega_prev[o];
            const double th = y[k * UT_THREADS];
            Theta[o] = th;
            const double d1 = om - th;
            const double xn = x + d1;               // X += Omega - Theta
            X[o] = xn;
            const double d2 = om - pv;
            acc[0] += w * (om * om); acc[1] += w * (th * th); acc[2] += w * (xn * xn);
            acc[3] += w * (d1 * d1); acc[4] += w * (d2 * d2);
        }
    }
    gg_block_sum<GG_NPART>(acc, scratch);
    if (threadIdx.x == 0) {
        double* out = partials + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * GG_NPART;
#pragma unroll
        for (int q = 0; q < GG_NPART; ++q) out[q] = acc[q];
    }
}

// A[m][j][i] = A[m][i][j] for i < j, for two stacks at once (Theta and X after the upper-triangle loop).
// One CTA per 32 x 32 tile pair (I <= J): coalesced read of tile (I,J), transposed through shared memory, coalesced
// write of tile (J,I).
__global__ void __launch_bounds__(256)
mirror_upper_kernel(double* __restrict__ A0, double* __restrict__ A1, int p)
{
    __shared__ double t[32][33];
    const int nt = (p + 31) / 32;
    int rem = blockIdx.x, I = 0;
    while (rem >= nt - I) { rem -= nt - I; ++I; }
    const int J = I + rem;
    double* A = (blockIdx.z ? A1 : A0) + (size_t)blockIdx.y * p * p;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int i = I * 32 + r, j = J * 32 + tx;
        if (i < p && j < p) t[r][tx] = A[(size_t)i * p + j];
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int i = J * 32 + r, j = I * 32 + tx;          // entry (i,j) of the mirror tile = t[tx][r]
        if (i < p && j < p && i > j) A[(size_t)i * p + j] = t[tx][r];
    }
}

// ------------------------------------------------------------------------------------------
// Stopping test + rho update, one CTA per problem; deterministic (fixed-order) reduction.
__global__ void __launch_bounds__(256)
stop_update_kernel(const double* __restrict__ partials, int nparts, double* __restrict__ ctrl,
                   double* __restrict__ hist, int hist_cap, const double* __restrict__ pdim,
                   double tol, double rtol, int update_rho)
{
    __shared__ double scratch[GG_NPART * 32];
    const int q = blockIdx.x;
    double* c = ctrl + (size_t)q * GG_CTRL_STRIDE;
    if (c[GG_C_DONE] != 0.0) return;
    const double* P = partials + (size_t)q * nparts * GG_NPART;
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int t = threadIdx.x; t < nparts; t += blockDim.x) {
#pragma unroll
        for (int i = 0; i < GG_NPART; ++i) acc[i] += P[(size_t)t * GG_NPART + i];
    }
    gg_block_sum<GG_NPART>(acc, scratch);
    if (threadIdx.x == 0) {
        const double rho = c[GG_C_RHO];
        const double nO = sqrt(acc[0]), nTL = sqrt(acc[1]), nX = sqrt(acc[2]);
        const double r = sqrt(acc[3]);
        const double s = rho * sqrt(acc[4]);
        const double dim = pdim[q];
        const double e_pri = dim * tol + rtol * fmax(nO, nTL);
        const double e_dual = dim * tol + rtol * rho * nX;
        const int it = (int)c[GG_C_ITER];
        if (it < hist_cap) {
            double* h = hist + ((size_t)q * hist_cap + it) * GG_HIST_STRIDE;
            h[0] = r; h[1] = s; h[2] = e_pri; h[3] = e_dual; h[4] = rho;
        }
        double rho_new = rho;
        if (update_rho) {
            if (r >= 10.0 * s) rho_new = 2.0 * rho;
            else if (s >= 10.0 * r) rho_new = 0.5 * rho;
        }
        c[GG_C_XSCALE] = rho / rho_new;
        c[GG_C_RHO] = rho_new;
        c[GG_C_R] = r; c[GG_C_S] = s; c[GG_C_EPRI] = e_pri; c[GG_C_EDUAL] = e_dual;
        c[GG_C_ITER] = (double)(it + 1);
        if (r <= e_pri && s <= e_dual) { c[GG_C_STATUS] = 1.0; c[GG_C_DONE] = 1.0; }
        // a non-finite iterate (non-finite input, or an eigendecomposition that broke down) stops the problem with
        // status -1; the host turns it into an exception, as numpy's eigh would (LinAlgError)
        if (!(isfinite(r) && isfinite(s))) { c[GG_C_STATUS] = -1.0; c[GG_C_DONE] = 1.0; }
    }
}

// X *= pending scale (applied once after the loop; inside the loop build_w folds it in).
__global__ void __launch_bounds__(EW_THREADS)
scale_pending_kernel(double* __restrict__ X, double* __restrict__ ctrl, int mpp, size_t pp)
{
    const int m = blockIdx.y;
    const double xs = ctrl[(size_t)(m / mpp) * GG_CTRL_STRIDE + GG_C_XSCALE];
    if (xs == 1.0) return;
    const size_t base = (size_t)m * pp;
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS)
        X[base + e] = xs * X[base + e];
}

__global__ void reset_xscale_kernel(double* ctrl, int nprob)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nprob) ctrl[(size_t)q * GG_CTRL_STRIDE + GG_C_XSCALE] = 1.0;
}

// ------------------------------------------------------------------------------------------
// Objective pieces (measure=True): <Omega,S>, and the regulariser P(Theta) on the strict upper
// triangle (ggl_helper.py:162-176).  out[0] += <Omega,S>, out[1] += 2*sum(l1*|.|_1 + l2*(|.|_2 or TV)).
__global__ void __launch_bounds__(EW_THREADS)
objective_kernel(const double* __restrict__ Omega, const double* __restrict__ S, const double* __restrict__ Theta,
                 double lambda1, double lambda2, int reg, int K, int p, double* __restrict__ partials)
{
    __shared__ double scratch[2 * 32];
    const size_t pp = (size_t)p * p;
    double acc[2] = {0.0, 0.0};
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        double n1 = 0.0, n2 = 0.0, prev = 0.0;
        for (int k = 0; k < K; ++k) {
            acc[0] += Omega[k * pp + e] * S[k * pp + e];
            if (j > i && reg >= 0) {
                const double a = Theta[k * pp + e];
                n1 += fabs(a);
                if (reg == 0) n2 += a * a;
                else if (k > 0) n2 += fabs(a - prev);
                prev = a;
            }
        }
        if (j > i && reg >= 0) {
            if (reg == 0) n2 = sqrt(n2);
            acc[1] += lambda1 * n1 + lambda2 * n2;
        }
    }
    gg_block_sum<2>(acc, scratch);
    if (threadIdx.x == 0) {
        partials[2 * blockIdx.x] = acc[0];
        partials[2 * blockIdx.x + 1] = 2.0 * acc[1];
    }
}

// max |A - A^T| per stack (symmetry check after the loop: admm_solver.py:284-291)
__global__ void __launch_bounds__(EW_THREADS)
asym_max_kernel(const double* __restrict__ A, int p, double* __restrict__ out)
{
    __shared__ double scratch[32];
    const int m = blockIdx.y;
    const size_t pp = (size_t)p * p;
    const double* a = A + (size_t)m * pp;
    double mx = 0.0;
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        if (j > i) mx = fmax(mx, fabs(a[e] - a[(size_t)j * p + i]));
    }
    mx = gg_block_max(mx, scratch);
    if (threadIdx.x == 0) out[(size_t)m * gridDim.x + blockIdx.x] = mx;
}

// ------------------------------------------------------------------------------------------
// K-sharded MGL (one process per GPU): V = (Omega + L) + X is exchanged from instance layout to row-band
// layout, the cross-instance prox runs on the band, Theta travels back.
__global__ void __launch_bounds__(EW_THREADS)
add3_kernel(const double* __restrict__ Omega, const double* __restrict__ L, const double* __restrict__ X,
            double* __restrict__ V, size_t total)
{
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * EW_THREADS) {
        double v = Omega[e];
        if (L) v = v + L[e];
        V[e] = v + X[e];
    }
}

// Row-band bookkeeping of the K-sharded solve: the p rows are cut into `world` contiguous bands (the first p % world
// bands one row longer -- parallel.partition()); band d of this rank's K_loc instances is one contiguous block
// [K_loc][rows_d][p] of the all-to-all buffers, at offset K_loc * p * lo_d.
__device__ __forceinline__ size_t gg_band_offset(int m, int r, int c, int p, int K_loc, int world)
{
    const int base = p / world, rem = p - base * world, cut = rem * (base + 1);
    const int d = r < cut ? r / (base + 1) : rem + (r - cut) / base;
    const int lo = d < rem ? d * (base + 1) : cut + (d - rem) * base;
    const int rows = base + (d < rem ? 1 : 0);
    return (size_t)K_loc * p * lo + ((size_t)m * rows + (r - lo)) * p + c;
}

// send = (Omega + L) + X written straight into the send buffer of the first all-to-all (one pass, no torch.cat)
__global__ void __launch_bounds__(EW_THREADS)
pack_bands_kernel(const double* __restrict__ Omega, const double* __restrict__ L, const double* __restrict__ X,
                  const double* __restrict__ ctrl, int p, int K_loc, int world, double* __restrict__ send)
{
    if (ctrl && ctrl[GG_C_DONE] != 0.0) return;
    const int m = blockIdx.y;
    const size_t pp = (size_t)p * p, base = (size_t)m * pp;
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int r = (int)(e / p), c = (int)(e - (size_t)r * p);
        double v = Omega[base + e];
        if (L) v = v + L[base + e];
        send[gg_band_offset(m, r, c, p, K_loc, world)] = v + X[base + e];
    }
}

// Theta arrives in the receive buffer of the second all-to-all (same block layout as the send buffer above): one
// pass writes Theta in instance layout and either C = Theta - X - Omega (latent) or the dual update
// X += Omega - Theta with the five residual partial sums (same expressions as prox_mgl_kernel's phase B).
__global__ void __launch_bounds__(EW_THREADS)
unpack_dual_kernel(const double* __restrict__ recv, const double* __restrict__ Omega,
                   const double* __restrict__ Omega_prev, double* __restrict__ X, double* __restrict__ Theta,
                   double* __restrict__ C, const double* __restrict__ ctrl, int p, int K_loc, int world,
                   double* __restrict__ partials)
{
    __shared__ double scratch[GG_NPART * 32];
    if (ctrl[GG_C_DONE] != 0.0) return;
    const int m = blockIdx.y;
    const size_t pp = (size_t)p * p, base = (size_t)m * pp;
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int r = (int)(e / p), c = (int)(e - (size_t)r * p);
        const double th = recv[gg_band_offset(m, r, c, p, K_loc, world)];
        const double om = Omega[base + e], x = X[base + e];
        Theta[base + e] = th;
        if (C) {
            C[base + e] = (th - x) - om;
        } else {
            const double d1 = om - th;
            const double xn = x + d1;
            X[base + e] = xn;
            const double d2 = om - Omega_prev[base + e];
            acc[0] += om * om; acc[1] += th * th; acc[2] += xn * xn; acc[3] += d1 * d1; acc[4] += d2 * d2;
        }
    }
    if (!C) {
        gg_block_sum<GG_NPART>(acc, scratch);
        if (threadIdx.x == 0) {
            double* out = partials + ((size_t)m * gridDim.x + blockIdx.x) * GG_NPART;
#pragma unroll
            for (int q = 0; q < GG_NPART; ++q) out[q] = acc[q];
        }
    }
}

// V, Theta: (K, nb, p) slabs holding global rows row0..row0+nb-1 of every instance.  One thread per entry;
// the K-vector lives in shared memory ([k][tid]: conflict free).  Every entry is computed from its own
// inputs, so with symmetric inputs the assembled Theta is symmetric and identical to prox_mgl_kernel's.
template <int REG>
__global__ void __launch_bounds__(256)
prox_band_kernel(const double* __restrict__ V, double* __restrict__ Theta, const double* __restrict__ ctrl,
                 double lambda1, double lambda2, int K, int nb, int p, int row0)
{
    extern __shared__ double ysm[];              // K * blockDim.x  (block size shrinks for large K)
    if (ctrl[GG_C_DONE] != 0.0) return;
    const double inv_rho = 1.0 / ctrl[GG_C_RHO];
    if (ctrl[GG_C_LAM1] > 0.0) { lambda1 = ctrl[GG_C_LAM1]; lambda2 = ctrl[GG_C_LAM2]; }
    const double l1 = inv_rho * lambda1, l2 = inv_rho * lambda2;
    const int T = blockDim.x;
    const size_t slab = (size_t)nb * p;
    const size_t e = (size_t)blockIdx.x * T + threadIdx.x;
    if (e >= slab) return;
    const int r = (int)(e / p), c = (int)(e - (size_t)r * p);
    double* y = ysm + threadIdx.x;
#pragma unroll 4
    for (int k = 0; k < K; ++k) y[k * T] = V[k * slab + e];
    if (row0 + r != c) {
        if (REG == 0) {
            double ss = 0.0;
            for (int k = 0; k < K; ++k) {
                const double u = gg_soft(y[k * T], l1);
                y[k * T] = u;
                ss += u * u;
            }
            const double nrm = sqrt(ss);
            const double a = nrm > l2 ? nrm : l2;
            const double f = a - l2;
            for (int k = 0; k < K; ++k) y[k * T] = (y[k * T] * f) / a;
        } else {
            gg_tv1d_inplace(y, K, T, l2);
            for (int k = 0; k < K; ++k) y[k * T] = gg_soft(y[k * T], l1);
        }
    }
#pragma unroll 4
    for (int k = 0; k < K; ++k) Theta[k * slab + e] = y[k * T];
}

// ------------------------------------------------------------------------------------------
// Peer-memory variants of the two exchange steps of the K-sharded loop (one process per GPU, buffers in symmetric
// memory, peer pointers mapped over NVLink): the kernels store straight into the receive buffers of the other ranks,
// so the re-tile IS the exchange -- no send buffer, no all-to-all; the host only puts a cross-rank barrier after each.
#define GG_MAX_PEERS 16
struct GgPeers { double* ptr[GG_MAX_PEERS]; };

__device__ __forceinline__ void gg_part(int n, int world, int idx, int& lo, int& len)
{   // parallel.partition(): the first n % world parts are one longer
    const int base = n / world, rem = n - base * world;
    lo = idx < rem ? idx * (base + 1) : rem * (base + 1) + (idx - rem) * base;
    len = base + (idx < rem ? 1 : 0);
}

// band buffer of rank d: (K_total, rows_d, p).  This rank's instances are k_lo .. k_lo + K_loc - 1.
__global__ void __launch_bounds__(EW_THREADS)
pack_bands_p2p_kernel(const double* __restrict__ Omega, const double* __restrict__ L, const double* __restrict__ X,
                      const double* __restrict__ ctrl, int p, int K_loc, int world, int k_lo, GgPeers band)
{
    if (ctrl && ctrl[GG_C_DONE] != 0.0) return;
    const int m = blockIdx.y;
    const size_t pp = (size_t)p * p, base = (size_t)m * pp;
    const int rb = p / world, rem = p - rb * world, cut = rem * (rb + 1);
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int r = (int)(e / p), c = (int)(e - (size_t)r * p);
        const int d = r < cut ? r / (rb + 1) : rem + (r - cut) / rb;
        const int lo = d < rem ? d * (rb + 1) : cut + (d - rem) * rb;
        const int rows = rb + (d < rem ? 1 : 0);
        double v = Omega[base + e];
        if (L) v = v + L[base + e];
        band.ptr[d][((size_t)(k_lo + m) * rows + (r - lo)) * p + c] = v + X[base + e];
    }
}

// prox on the local band (K, nb, p) of all instances; Theta of instance k goes to its owner's `back` buffer, which is
// laid out like the send / receive buffers of the all-to-all version: [band d][m][row][col], band d at offset
// K_loc(owner) * p * row0_d.
template <int REG>
__global__ void __launch_bounds__(256)
prox_band_p2p_kernel(const double* __restrict__ V, GgPeers back, const double* __restrict__ ctrl, double lambda1,
                     double lambda2, int K, int nb, int p, int row0, int world)
{
    extern __shared__ double ysm[];              // K * blockDim.x doubles
    if (ctrl[GG_C_DONE] != 0.0) return;
    const double inv_rho = 1.0 / ctrl[GG_C_RHO];
    if (ctrl[GG_C_LAM1] > 0.0) { lambda1 = ctrl[GG_C_LAM1]; lambda2 = ctrl[GG_C_LAM2]; }
    const double l1 = inv_rho * lambda1, l2 = inv_rho * lambda2;
    const int T = blockDim.x;
    const size_t slab = (size_t)nb * p;
    const size_t e = (size_t)blockIdx.x * T + threadIdx.x;
    if (e >= slab) return;
    const int r = (int)(e / p), c = (int)(e - (size_t)r * p);
    double* y = ysm + threadIdx.x;
#pragma unroll 4
    for (int k = 0; k < K; ++k) y[k * T] = V[k * slab + e];
    if (row0 + r != c) {
        if (REG == 0) {
            double ss = 0.0;
            for (int k = 0; k < K; ++k) {
                const double u = gg_soft(y[k * T], l1);
                y[k * T] = u;
                ss += u * u;
            }
            const double nrm = sqrt(ss);
            const double a = nrm > l2 ? nrm : l2;
            const double f = a - l2;
            for (int k = 0; k < K; ++k) y[k * T] = (y[k * T] * f) / a;
        } else {
            gg_tv1d_inplace(y, K, T, l2);
            for (int k = 0; k < K; ++k) y[k * T] = gg_soft(y[k * T], l1);
        }
    }
    for (int s = 0; s < world; ++s) {
        int k0, kl;
        gg_part(K, world, s, k0, kl);
        double* dst = back.ptr[s] + (size_t)kl * p * row0 + e;
        for (int m = 0; m < kl; ++m) dst[(size_t)m * slab] = y[(k0 + m) * T];
    }
}

// ------------------------------------------------------------------------------------------
// ext_ADMM_MGL (non-conforming group graphical lasso, src/gglasso/solver/ext_admm_solver.py:191-273).
// The K matrices of different size p_k are padded to a common p (decoupled unit diagonal, see block_SGL);
// pvec[k] = p_k masks the padding out of the norms.  One ADMM problem, rho fixed.
//
// Theta update: V = (Omega + L + X0 + Lambda - X1)/2, Theta = prox_od_1norm(V, lambda1_k/(2 rho))   (:206-208)
// latent: C = Theta - X0 - Omega                                                                   (:212-216)
__global__ void __launch_bounds__(EW_THREADS)
ext_theta_kernel(const double* __restrict__ Omega, const double* __restrict__ L, const double* __restrict__ X0,
                 const double* __restrict__ Lam, const double* __restrict__ X1, const double* __restrict__ lam1,
                 const double* __restrict__ ctrl, int p, double* __restrict__ Theta, double* __restrict__ C)
{
    if (ctrl[GG_C_DONE] != 0.0) return;
    const int m = blockIdx.y;
    const double thr = lam1[m] / (2.0 * ctrl[GG_C_RHO]);
    const size_t pp = (size_t)p * p, base = (size_t)m * pp;
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        const double om = Omega[base + e], x0 = X0[base + e];
        double v = om;
        if (L) v = v + L[base + e];
        v = v + x0;
        v = v + Lam[base + e];
        v = (v - X1[base + e]) * 0.5;
        const double th = (i == j) ? v : gg_soft(v, thr);
        Theta[base + e] = th;
        if (C) C[base + e] = (th - x0) - om;
    }
}

// Lambda = prox_2norm_G(Theta + X1, G, lambda2/rho)   (:219-223, :394-453).  Step 1 copies Z = Theta + X1;
// step 2: one thread per group l gathers the member entries (G[0,l,k], G[1,l,k]) != -1 over k, shrinks the
// vector in Euclidean norm with threshold (lambda2/rho) sqrt(group size) and scatters it to (i,j) and (j,i).
__global__ void __launch_bounds__(EW_THREADS)
ext_z_kernel(const double* __restrict__ Theta, const double* __restrict__ X1, const double* __restrict__ ctrl,
             size_t total, double* __restrict__ Z)
{
    if (ctrl[GG_C_DONE] != 0.0) return;
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * EW_THREADS)
        Z[e] = Theta[e] + X1[e];
}

__global__ void __launch_bounds__(128)
ext_group_prox_kernel(const double* __restrict__ Theta, const double* __restrict__ X1, const int* __restrict__ G,
                      int Lg, int K, int p, double lambda2, const double* __restrict__ ctrl, double* __restrict__ Lam)
{
    if (ctrl[GG_C_DONE] != 0.0) return;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Lg) return;
    const size_t pp = (size_t)p * p;
    const int* Gi = G + (size_t)l * K;                 // G[0,l,:]
    const int* Gj = G + (size_t)Lg * K + (size_t)l * K;  // G[1,l,:]
    double ss = 0.0;
    int cnt = 0;
    for (int k = 0; k < K; ++k) {
        const int i = Gi[k];
        if (i < 0) continue;
        const size_t e = (size_t)k * pp + (size_t)i * p + Gj[k];
        const double v = Theta[e] + X1[e];
        ss += v * v;
        ++cnt;
    }
    const double lam = (lambda2 / ctrl[GG_C_RHO]) * sqrt((double)cnt);
    const double nrm = sqrt(ss);
    const double a = nrm > lam ? nrm : lam;
    for (int k = 0; k < K; ++k) {
        const int i = Gi[k];
        if (i < 0) continue;
        const int j = Gj[k];
        const size_t e = (size_t)k * pp + (size_t)i * p + j;
        const double v = Theta[e] + X1[e];
        const double z = (v * (a - lam)) / a;
        Lam[e] = z;
        Lam[(size_t)k * pp + (size_t)j * p + i] = z;
    }
}

// X0 += Omega - Theta + L ; X1 += Theta - Lambda ; residual partial sums of the ext criterion (:330-347):
//   [0] |Omega|^2+|Lambda|^2  [1] |Theta-L|^2+|Theta|^2  [2] |X0|^2+|X1|^2
//   [3] |Omega-Theta+L|^2+|Lambda-Theta|^2  [4] |Omega-Omega_prev|^2+|Lambda-Lambda_prev|^2
__global__ void __launch_bounds__(EW_THREADS)
ext_dual_kernel(double* __restrict__ X0, double* __restrict__ X1, const double* __restrict__ Omega,
                const double* __restrict__ Omega_prev, const double* __restrict__ Theta, const double* __restrict__ L,
                const double* __restrict__ Lam, const double* __restrict__ Lam_prev, const double* __restrict__ ctrl,
                const int* __restrict__ pvec, int p, double* __restrict__ partials)
{
    __shared__ double scratch[GG_NPART * 32];
    if (ctrl[GG_C_DONE] != 0.0) return;
    const int m = blockIdx.y;
    const int pb = pvec ? pvec[m] : p;
    const size_t pp = (size_t)p * p, base = (size_t)m * pp;
    double acc[GG_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (size_t e = (size_t)blockIdx.x * EW_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * EW_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        const double om = Omega[base + e], th = Theta[base + e], la = Lam[base + e];
        const double l = L ? L[base + e] : 0.0;
        const double r0 = L ? ((om - th) + l) : (om - th);
        const double r1 = th - la;
        const double x0 = X0[base + e] + r0, x1 = X1[base + e] + r1;
        X0[base + e] = x0;
        X1[base + e] = x1;
        if (i < pb && j < pb) {
            const double tl = th - l, d0 = om - Omega_prev[base + e], d1 = la - Lam_prev[base + e];
            acc[0] += om * om + la * la;
            acc[1] += tl * tl + th * th;
            acc[2] += x0 * x0 + x1 * x1;
            acc[3] += r0 * r0 + r1 * r1;
            acc[4] += d0 * d0 + d1 * d1;
        }
    }
    gg_block_sum<GG_NPART>(acc, scratch);
    if (threadIdx.x == 0) {
        double* out = partials + ((size_t)m * gridDim.x + blockIdx.x) * GG_NPART;
#pragma unroll
        for (int q = 0; q < GG_NPART; ++q) out[q] = acc[q];
    }
}

// ==========================================================================================
// host launchers (C++ linkage; the extern "C" ABI lives in gg_capi.cu)
// ==========================================================================================
static inline int ew_blocks(size_t pp, int M)
{
    // enough CTAs to fill 148 SMs x 8 resident CTAs, but no more than the work needs
    size_t need = (pp + (size_t)EW_THREADS * EW_UNROLL - 1) / ((size_t)EW_THREADS * EW_UNROLL);
    size_t cap = (size_t)(148 * 8 + M - 1) / M;
    if (cap < 1) cap = 1;
    size_t b = need < cap ? need : cap;
    return (int)(b < 1 ? 1 : b);
}

int gg_launch_build_w(const double* Theta, const double* L, double* X, const double* S, const double* nk,
                      const double* ctrl, int M, int p, int mpp, double* W, cudaStream_t st)
{
    const size_t pp = (size_t)p * p;
    dim3 grid(ew_blocks(pp, M), M);
    gg_count_launch(1);
    build_w_kernel<<<grid, EW_THREADS, 0, st>>>(Theta, L, X, S, nk, ctrl, mpp, pp, W);
    GG_CHECK_LAUNCH();
    return 0;
}

extern "C" int gg_sgl_nparts(int p, int M) { return ew_blocks((size_t)p * p, M); }

int gg_launch_prox_sgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                       double* C, const double* ctrl, double lam, const double* lam_mat, int M, int p,
                       double* partials, const int* pvec, double* blk_nrm, int Mblk, cudaStream_t st)
{
    dim3 grid(gg_sgl_nparts(p, M), M);
    if (blk_nrm) {
        if (Mblk <= 0 || p % Mblk != 0) return -1;
        const int nbk = p / Mblk;
        dim3 gn((nbk * nbk + 7) / 8, M);
        gg_count_launch(1);
        fsgl_block_norm_kernel<<<gn, 256, 0, st>>>(Omega, L, X, ctrl, p, Mblk, blk_nrm);
    }
    gg_count_launch(1);
    prox_sgl_kernel<<<grid, EW_THREADS, 0, st>>>(Omega, Omega_prev, L, X, Theta, C, ctrl, lam, lam_mat, p, partials,
                                                 pvec, blk_nrm, Mblk);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_dual_update(double* X, const double* Omega, const double* Omega_prev, const double* Theta,
                          const double* L, const double* ctrl, int M, int p, int mpp, int sgl_order,
                          double* partials, cudaStream_t st)
{
    const size_t pp = (size_t)p * p;
    dim3 grid(gg_sgl_nparts(p, M), M);
    gg_count_launch(1);
    dual_update_kernel<<<grid, EW_THREADS, 0, st>>>(X, Omega, Omega_prev, Theta, L, ctrl, mpp, pp, sgl_order, partials);
    GG_CHECK_LAUNCH();
    return 0;
}

extern "C" int gg_mgl_ntile(int p) { return (p + PT - 1) / PT; }

template <int REG, bool LATENT>
static int launch_prox_mgl_t(const double* Omega, const double* Omega_prev, const double* L, double* X,
                             double* Theta, double* C, const double* ctrl, double l1, double l2, int K, int p,
                             int nprob, double* partials, cudaStream_t st)
{
    const int nt = gg_mgl_ntile(p);
    const size_t smem = (size_t)K * PSLOT * sizeof(double);
    if (smem > 200 * 1024) return -2;   // K too large for the shared-memory layout
    auto kern = prox_mgl_kernel<REG, LATENT>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    const int nst = (nt + 3) / 4;
    dim3 grid(16 * (nst * (nst + 1) / 2), nprob);
    gg_count_launch(1);
    kern<<<grid, PT * PT, smem, st>>>(Omega, Omega_prev, L, X, Theta, C, ctrl, l1, l2, K, p, partials);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_prox_mgl(const double* Omega, const double* Omega_prev, const double* L, double* X, double* Theta,
                       double* C, const double* ctrl, double l1, double l2, int reg, int K, int p, int nprob,
                       double* partials, cudaStream_t st)
{
    const bool latent = (C != nullptr);
    if (reg == 0) {
        return latent ? launch_prox_mgl_t<0, true>(Omega, Omega_prev, L, X, Theta, C, ctrl, l1, l2, K, p, nprob, partials, st)
                      : launch_prox_mgl_t<0, false>(Omega, Omega_prev, L, X, Theta, C, ctrl, l1, l2, K, p, nprob, partials, st);
    }
    return latent ? launch_prox_mgl_t<1, true>(Omega, Omega_prev, L, X, Theta, C, ctrl, l1, l2, K, p, nprob, partials, st)
                  : launch_prox_mgl_t<1, false>(Omega, Omega_prev, L, X, Theta, C, ctrl, l1, l2, K, p, nprob, partials, st);
}

int gg_launch_prox_mgl_ragged(const double* Omega, const double* Omega_prev, double* X, double* Theta,
                              const double* ctrl, double l1, double l2, int reg, int K, int p, int nprob,
                              const int* pvec, double* partials, cudaStream_t st)
{
    const int nt = gg_mgl_ntile(p);
    const size_t smem = (size_t)K * PSLOT * sizeof(double);
    if (smem > 200 * 1024) return -2;   // K too large for the shared-memory layout
    auto kern = reg == 0 ? prox_mgl_ragged_kernel<0> : prox_mgl_ragged_kernel<1>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    const int nst = (nt + 3) / 4;
    dim3 grid(16 * (nst * (nst + 1) / 2), nprob);
    gg_count_launch(1);
    kern<<<grid, PT * PT, smem, st>>>(Omega, Omega_prev, X, Theta, ctrl, l1, l2, K, p, pvec, partials);
    GG_CHECK_LAUNCH();
    return 0;
}

extern "C" int gg_mgl_upper_nparts(int p) { return ut_ntiles(p); }

int gg_launch_prox_mgl_upper(const double* Omega, const double* Omega_prev, double* X, double* Theta,
                             const double* ctrl, double l1, double l2, int reg, int K, int p, int nprob,
                             double* partials, cudaStream_t st)
{
    const size_t smem = (size_t)K * UT_THREADS * sizeof(double);
    if (smem > 200 * 1024) return -2;   // K too large for the shared-memory layout
    auto kern = reg == 0 ? prox_mgl_upper_kernel<0> : prox_mgl_upper_kernel<1>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    gg_count_launch(1);
    kern<<<dim3(ut_ntiles(p), nprob), UT_THREADS, smem, st>>>(Omega, Omega_prev, X, Theta, ctrl, l1, l2, K, p,
                                                              partials);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_build_w_upper(const double* Theta, double* X, const double* S, const double* nk, const double* ctrl,
                            int K, int p, int nprob, double* W, cudaStream_t st)
{
    dim3 grid((p + 1) / 2, K, nprob);
    gg_count_launch(1);
    build_w_upper_kernel<<<grid, EW_THREADS, 0, st>>>(Theta, X, S, nk, ctrl, p, W);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_mirror_upper(double* A0, double* A1, int M, int p, cudaStream_t st)
{
    const int nt = (p + 31) / 32;
    dim3 grid(nt * (nt + 1) / 2, M, A1 ? 2 : 1);
    gg_count_launch(1);
    mirror_upper_kernel<<<grid, 256, 0, st>>>(A0, A1, p);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_stop_update(const double* partials, int nparts, double* ctrl, double* hist, int hist_cap,
                          const double* pdim, double tol, double rtol, int update_rho, int nprob, cudaStream_t st)
{
    gg_count_launch(1);
    stop_update_kernel<<<nprob, 256, 0, st>>>(partials, nparts, ctrl, hist, hist_cap, pdim, tol, rtol, update_rho);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_scale_pending(double* X, double* ctrl, int M, int p, int mpp, cudaStream_t st)
{
    const size_t pp = (size_t)p * p;
    dim3 grid(ew_blocks(pp, M), M);
    gg_count_launch(1);
    scale_pending_kernel<<<grid, EW_THREADS, 0, st>>>(X, ctrl, mpp, pp);
    GG_CHECK_LAUNCH();
    const int nprob = M / mpp;
    gg_count_launch(1);
    reset_xscale_kernel<<<(nprob + 127) / 128, 128, 0, st>>>(ctrl, nprob);
    GG_CHECK_LAUNCH();
    return 0;
}

extern "C" int gg_objective_nparts(int p) { return ew_blocks((size_t)p * p, 1); }

int gg_launch_objective(const double* Omega, const double* S, const double* Theta, double l1, double l2, int reg,
                        int K, int p, double* partials, cudaStream_t st)
{
    gg_count_launch(1);
    objective_kernel<<<gg_objective_nparts(p), EW_THREADS, 0, st>>>(Omega, S, Theta, l1, l2, reg, K, p, partials);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_asym_max(const double* A, int M, int p, double* out, cudaStream_t st)
{
    dim3 grid(gg_sgl_nparts(p, M), M);
    gg_count_launch(1);
    asym_max_kernel<<<grid, EW_THREADS, 0, st>>>(A, p, out);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_add3(const double* Omega, const double* L, const double* X, double* V, size_t total, cudaStream_t st)
{
    size_t blocks = (total + EW_THREADS - 1) / EW_THREADS;
    if (blocks > 148 * 16) blocks = 148 * 16;
    gg_count_launch(1);
    add3_kernel<<<(unsigned)blocks, EW_THREADS, 0, st>>>(Omega, L, X, V, total);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_pack_bands(const double* Omega, const double* L, const double* X, const double* ctrl, int K_loc, int p,
                         int world, double* send, cudaStream_t st)
{
    dim3 grid(gg_sgl_nparts(p, K_loc), K_loc);
    gg_count_launch(1);
    pack_bands_kernel<<<grid, EW_THREADS, 0, st>>>(Omega, L, X, ctrl, p, K_loc, world, send);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_unpack_dual(const double* recv, const double* Omega, const double* Omega_prev, double* X, double* Theta,
                          double* C, const double* ctrl, int K_loc, int p, int world, double* partials,
                          cudaStream_t st)
{
    dim3 grid(gg_sgl_nparts(p, K_loc), K_loc);
    gg_count_launch(1);
    unpack_dual_kernel<<<grid, EW_THREADS, 0, st>>>(recv, Omega, Omega_prev, X, Theta, C, ctrl, p, K_loc, world, partials);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_prox_band(const double* V, double* Theta, const double* ctrl, double l1, double l2, int reg, int K,
                        int nb, int p, int row0, cudaStream_t st)
{
    // the K-vector of every entry lives in shared memory: shrink the block until K*T*8 fits (~96 KB keeps two
    // CTAs per SM); K up to ~3000 is supported with 32-thread blocks
    int T = 256;
    while (T > 32 && (size_t)K * T * sizeof(double) > 96 * 1024) T >>= 1;
    const size_t smem = (size_t)K * T * sizeof(double);
    if (smem > 200 * 1024) return -2;
    const size_t slab = (size_t)nb * p;
    const unsigned grid = (unsigned)((slab + T - 1) / T);
    if (grid == 0) return 0;
    if (reg == 0) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(prox_band_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gg_count_launch(1);
        prox_band_kernel<0><<<grid, T, smem, st>>>(V, Theta, ctrl, l1, l2, K, nb, p, row0);
    } else {
        if (smem > 48 * 1024) cudaFuncSetAttribute(prox_band_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gg_count_launch(1);
        prox_band_kernel<1><<<grid, T, smem, st>>>(V, Theta, ctrl, l1, l2, K, nb, p, row0);
    }
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_pack_bands_p2p(const double* Omega, const double* L, const double* X, const double* ctrl, int K_loc,
                             int p, int world, int k_lo, double* const* peer_band, cudaStream_t st)
{
    GgPeers pb;
    for (int i = 0; i < GG_MAX_PEERS; ++i) pb.ptr[i] = i < world ? peer_band[i] : nullptr;
    dim3 grid(gg_sgl_nparts(p, K_loc), K_loc);
    gg_count_launch(1);
    pack_bands_p2p_kernel<<<grid, EW_THREADS, 0, st>>>(Omega, L, X, ctrl, p, K_loc, world, k_lo, pb);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_prox_band_p2p(const double* V, double* const* peer_back, const double* ctrl, double l1, double l2, int reg,
                            int K, int nb, int p, int row0, int world, cudaStream_t st)
{
    GgPeers pb;
    for (int i = 0; i < GG_MAX_PEERS; ++i) pb.ptr[i] = i < world ? peer_back[i] : nullptr;
    int T = 256;
    while (T > 32 && (size_t)K * T * sizeof(double) > 96 * 1024) T >>= 1;
    const size_t smem = (size_t)K * T * sizeof(double);
    if (smem > 200 * 1024) return -2;
    const size_t slab = (size_t)nb * p;
    const unsigned grid = (unsigned)((slab + T - 1) / T);
    if (grid == 0) return 0;
    if (reg == 0) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(prox_band_p2p_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gg_count_launch(1);
        prox_band_p2p_kernel<0><<<grid, T, smem, st>>>(V, pb, ctrl, l1, l2, K, nb, p, row0, world);
    } else {
        if (smem > 48 * 1024) cudaFuncSetAttribute(prox_band_p2p_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gg_count_launch(1);
        prox_band_p2p_kernel<1><<<grid, T, smem, st>>>(V, pb, ctrl, l1, l2, K, nb, p, row0, world);
    }
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_ext_theta(const double* Omega, const double* L, const double* X0, const double* Lam, const double* X1,
                        const double* lam1, const double* ctrl, int K, int p, double* Theta, double* C, cudaStream_t st)
{
    dim3 grid(gg_sgl_nparts(p, K), K);
    gg_count_launch(1);
    ext_theta_kernel<<<grid, EW_THREADS, 0, st>>>(Omega, L, X0, Lam, X1, lam1, ctrl, p, Theta, C);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_ext_lambda(const double* Theta, const double* X1, const int* G, int Lg, int K, int p, double lambda2,
                         const double* ctrl, double* Lam, cudaStream_t st)
{
    const size_t total = (size_t)K * p * p;
    size_t blocks = (total + EW_THREADS - 1) / EW_THREADS;
    if (blocks > 148 * 16) blocks = 148 * 16;
    gg_count_launch(1);
    ext_z_kernel<<<(unsigned)blocks, EW_THREADS, 0, st>>>(Theta, X1, ctrl, total, Lam);
    GG_CHECK_LAUNCH();
    if (Lg > 0) {
        gg_count_launch(1);
        ext_group_prox_kernel<<<(Lg + 127) / 128, 128, 0, st>>>(Theta, X1, G, Lg, K, p, lambda2, ctrl, Lam);
        GG_CHECK_LAUNCH();
    }
    return 0;
}

int gg_launch_ext_dual(double* X0, double* X1, const double* Omega, const double* Omega_prev, const double* Theta,
                       const double* L, const double* Lam, const double* Lam_prev, const double* ctrl,
                       const int* pvec, int K, int p, double* partials, cudaStream_t st)
{
    dim3 grid(gg_sgl_nparts(p, K), K);
    gg_count_launch(1);
    ext_dual_kernel<<<grid, EW_THREADS, 0, st>>>(X0, X1, Omega, Omega_prev, Theta, L, Lam, Lam_prev, ctrl, pvec, p,
                                                 partials);
    GG_CHECK_LAUNCH();
    return 0;
}
