// gg_ppdna.cu -- kernels of the proximal point dual Newton method (PPDNA) for GGL / FGL (sm_100a).
//
// Replaces the numba/numpy second-order part of the reference (src/gglasso/solver/ppdna_solver.py PPA_subproblem:65,
// ggl_helper.py:74-159 Jacobians of prox_p, :218-249 eval_jacobian_prox_p, :323-357 construct_gamma /
// eval_jacobian_phiplus, :361-437 hessian_Y / cg_ppdna).  X is the unscaled dual; at one point of the subproblem
//
//   gg_ppdna_build     Xs = X + s dX,  W = Omega_t - sigma (S + Xs),  V = Theta_t + sigma Xs          (full matrices)
//   gg_ppdna_spectral  from Vt, d = eigh(W): Q = Vt^T, phi = phi(d), sum log phi, Omega = Vt^T diag(phi) Vt (DMMA)
//   gg_ppdna_prox      Theta = prox_p(V, sigma l1, sigma l2) with the device routines of gg_prox_mgl (bit-identical),
//                      the Jacobian data of prox_p, grad Phi = Theta - Omega and the partial sums of Phi
//   gg_ppdna_hess      H[D] = sigma (Q (Gamma o (Q^T D Q)) Q^T + J_P[D]), Gamma_ab = phi_a phi_b / (phi_a phi_b + sigma):
//                      four TN products on FP64 tensor cores (two of them symmetric: ~6 p^3 flops per matrix), Gamma
//                      formed in an epilogue, J_P and the sigma scaling in one elementwise pass
//   gg_ppdna_cg        CG iterations on H d = -grad with alpha, beta, |r|^2 and the stop flag in device memory
//
// Every kernel takes a done flag (may be NULL): once *flag != 0 it returns at once, so CG iterations enqueued after
// convergence are no-ops and the host only polls the flag every few iterations.
// Compiled with -fmad=false: the prox expressions must match gg_prox_mgl (gg_elementwise.cu) bit for bit.
#include "gg_common.cuh"
#include "gg_condat.cuh"

#define PD_THREADS 256
#define PD_MAXB 1184           // 148 SMs x 8 resident CTAs
#define PD_TT 64               // output tile of the DMMA products
#define PD_KC 16               // reduction chunk
#define PD_LD (PD_TT + 4)      // conflict-free fragment loads (as gg_recon.cu)
#define PD_PT 16               // prox tile
#define PD_PLD 17
#define PD_PSLOT (PD_PT * PD_PLD)
#define PD_NPART 6             // <S,Omega>, P(Theta), <X,Omega-Theta>, |Omega-Omega_t|^2, |Theta-Theta_t|^2, |grad|^2

// CG state (doubles, device): |r|^2, alpha, beta, done, iterations, tol^2, iteration cap, <p,Hp>
#define CG_RR 0
#define CG_ALPHA 1
#define CG_BETA 2
#define CG_DONE 3
#define CG_ITER 4
#define CG_TOL2 5
#define CG_CAP 6

__device__ __forceinline__ bool pd_done(const double* flag) { return flag != nullptr && *flag != 0.0; }

__device__ __forceinline__ double pd_phi(double d, double sigma)
{
    const double r = sqrt(d * d + 4.0 * sigma);
    return d >= 0.0 ? 0.5 * (d + r) : (2.0 * sigma) / (r - d);
}

static inline int pd_blocks(size_t n)
{
    size_t b = (n + PD_THREADS * 4 - 1) / (PD_THREADS * 4);
    if (b > PD_MAXB) b = PD_MAXB;
    return (int)(b < 1 ? 1 : b);
}

// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PD_THREADS)
pd_build_kernel(const double* __restrict__ Om_t, const double* __restrict__ Th_t, const double* __restrict__ S,
                const double* X, const double* __restrict__ dX, double s, double sigma, size_t n, double* Xs,
                double* __restrict__ W, double* __restrict__ V, const double* flag)
{
    if (pd_done(flag)) return;
    for (size_t e = (size_t)blockIdx.x * PD_THREADS + threadIdx.x; e < n; e += (size_t)gridDim.x * PD_THREADS) {
        double x = X[e];
        if (dX) x = x + s * dX[e];
        Xs[e] = x;
        W[e] = Om_t[e] - sigma * (S[e] + x);
        V[e] = Th_t[e] + sigma * x;
    }
}

// phi = phi(d) per eigenvalue and logdet[m] = sum_c log phi  (one CTA per matrix, fixed-order reduction)
__global__ void __launch_bounds__(PD_THREADS)
pd_phi_kernel(const double* __restrict__ D, double sigma, int p, double* __restrict__ phi, double* __restrict__ logdet,
              const double* flag)
{
    __shared__ double scratch[32];
    if (pd_done(flag)) return;
    const int m = blockIdx.x;
    double acc[1] = {0.0};
    for (int c = threadIdx.x; c < p; c += PD_THREADS) {
        const double f = pd_phi(D[(size_t)m * p + c], sigma);
        phi[(size_t)m * p + c] = f;
        acc[0] += log(f);
    }
    gg_block_sum<1>(acc, scratch);
    if (threadIdx.x == 0) logdet[m] = acc[0];
}

__global__ void __launch_bounds__(256)
pd_transpose_kernel(const double* __restrict__ A, int p, double* __restrict__ T, const double* flag)
{
    __shared__ double t[32][33];
    if (pd_done(flag)) return;
    const size_t base = (size_t)blockIdx.z * p * p;
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int i = i0 + r, j = j0 + threadIdx.x;
        if (i < p && j < p) t[r][threadIdx.x] = A[base + (size_t)i * p + j];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int i = j0 + r, j = i0 + threadIdx.x;
        if (i < p && j < p) T[base + (size_t)i * p + j] = t[threadIdx.x][r];
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// C[m] = A[m]^T diag(fA[m]) B[m]  ("TN": C[i][j] = sum_c fA[c] A[c][i] B[c][j]) on DMMA m8n8k4, batched over blockIdx.z.
// The tile and warp shapes of recon_kernel (64 x 64 per CTA, 16 x 32 per warp, cp.async double buffer).
// SYM: the product is symmetric; only tiles I <= J are computed and the mirror is written through shared memory, so
// the result is exactly symmetric.  GAMMA: the result is multiplied by Gamma_ij = phi_i phi_j / (phi_i phi_j + sigma).
template <bool SYM, bool GAMMA, bool VEC>
__global__ void __launch_bounds__(256)
pd_tn_kernel(const double* __restrict__ A, const double* __restrict__ fA, const double* __restrict__ B, int p,
             double* __restrict__ C, const double* __restrict__ phi, double sigma, const double* flag)
{
    __shared__ __align__(16) double sm[2 * 2 * PD_KC * PD_LD];   // As[2][KC][LD], Bs[2][KC][LD]; reused as Cs[64][65]
    __shared__ double fs[2][PD_KC];
    const int I = blockIdx.y, J = blockIdx.x, m = blockIdx.z;
    if (SYM && I > J) return;
    if (pd_done(flag)) return;
    const size_t pp = (size_t)p * p;
    const double* Am = A + (size_t)m * pp;
    const double* Bm = B + (size_t)m * pp;
    const double* fm = fA ? fA + (size_t)m * p : nullptr;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;
    const int wr = wid >> 1, wc = wid & 1;
    const int i0 = I * PD_TT, j0 = J * PD_TT;
    const int nchunks = (p + PD_KC - 1) / PD_KC;

    auto load_chunk = [&](int c, int buf) {
        double* As = sm + (size_t)buf * PD_KC * PD_LD;
        double* Bs = sm + (size_t)(2 + buf) * PD_KC * PD_LD;
        const int c0 = c * PD_KC;
        if (VEC) {
            for (int idx = tid; idx < 2 * PD_KC * (PD_TT / 2); idx += 256) {
                const int which = idx / (PD_KC * (PD_TT / 2));
                const int rem = idx % (PD_KC * (PD_TT / 2));
                const int kk = rem / (PD_TT / 2), e = (rem % (PD_TT / 2)) * 2;
                const int gc = (which ? j0 : i0) + e, gr = c0 + kk;
                double* dst = (which ? Bs : As) + kk * PD_LD + e;
                if (gr < p && gc < p) gg_cp_async16(dst, (which ? Bm : Am) + (size_t)gr * p + gc);
                else { dst[0] = 0.0; dst[1] = 0.0; }
            }
        } else {
            for (int idx = tid; idx < 2 * PD_KC * PD_TT; idx += 256) {
                const int which = idx / (PD_KC * PD_TT);
                const int rem = idx % (PD_KC * PD_TT);
                const int kk = rem / PD_TT, e = rem % PD_TT;
                const int gc = (which ? j0 : i0) + e, gr = c0 + kk;
                double* dst = (which ? Bs : As) + kk * PD_LD + e;
                if (gr < p && gc < p) gg_cp_async8(dst, (which ? Bm : Am) + (size_t)gr * p + gc);
                else dst[0] = 0.0;
            }
        }
        if (tid < PD_KC) {
            const int cc = c0 + tid;
            fs[buf][tid] = (cc < p) ? (fm ? fm[cc] : 1.0) : 0.0;
        }
        gg_cp_commit();
    };

    double acc[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }

    load_chunk(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) { load_chunk(c + 1, (c + 1) & 1); gg_cp_wait<1>(); }
        else gg_cp_wait<0>();
        __syncthreads();
        const int buf = c & 1;
        const double* As = sm + (size_t)buf * PD_KC * PD_LD;
        const double* Bs = sm + (size_t)(2 + buf) * PD_KC * PD_LD;
#pragma unroll
        for (int k0 = 0; k0 < PD_KC; k0 += 4) {
            const double f = fs[buf][k0 + fc];
            double fa[2], fb[4];
#pragma unroll
            for (int a = 0; a < 2; ++a) fa[a] = As[(k0 + fc) * PD_LD + (wr * 2 + a) * 8 + fr] * f;
#pragma unroll
            for (int b = 0; b < 4; ++b) fb[b] = Bs[(k0 + fc) * PD_LD + (wc * 4 + b) * 8 + fr];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) gg_dmma(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
        }
        __syncthreads();
    }

    double* Cs = sm;                         // 64 x 65
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int r = (wr * 2 + a) * 8 + fr, cc = (wc * 4 + b) * 8 + 2 * fc;
            Cs[r * 65 + cc] = acc[a][b][0];
            Cs[r * 65 + cc + 1] = acc[a][b][1];
        }
    __syncthreads();
    double* O = C + (size_t)m * pp;
    const double* ph = GAMMA ? phi + (size_t)m * p : nullptr;
    for (int idx = tid; idx < PD_TT * PD_TT; idx += 256) {
        const int r = idx / PD_TT, cc = idx % PD_TT;
        const int gi = i0 + r, gj = j0 + cc;
        if (gi < p && gj < p) {
            double v = (SYM && I == J && cc < r) ? Cs[cc * 65 + r] : Cs[r * 65 + cc];
            if (GAMMA) { const double q = ph[gi] * ph[gj]; v = v * (q / (q + sigma)); }
            O[(size_t)gi * p + gj] = v;
        }
    }
    if (SYM && I < J) {
        for (int idx = tid; idx < PD_TT * PD_TT; idx += 256) {
            const int r = idx / PD_TT, cc = idx % PD_TT;        // element (j0 + r, i0 + cc) of the mirror tile
            const int gi = j0 + r, gj = i0 + cc;
            if (gi < p && gj < p) {
                double v = Cs[cc * 65 + r];
                if (GAMMA) { const double q = ph[gi] * ph[gj]; v = v * (q / (q + sigma)); }
                O[(size_t)gi * p + gj] = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// prox_p of V + Jacobian data + gradient + partial sums of Phi.  One CTA per 16 x 16 tile pair (I <= J), thread
// (tr, tc) owns entry (I*16+tr, J*16+tc); the K-vector is processed in shared memory with exactly the expressions of
// prox_mgl_kernel (gg_elementwise.cu), phase B writes the tile and its mirror.
//   code[k][i][j]: bit 0 = GGL mask 1[|v| > sigma l1] resp. FGL active 1[|z| > sigma l1]; bit 1 = FGL run start
//   jscale[i][j]:  GGL sigma l2 / |u| (or -1 on the zero branch |u| <= sigma l2)
template <int REG>
__global__ void __launch_bounds__(PD_PT * PD_PT)
pd_prox_kernel(const double* __restrict__ V, const double* __restrict__ Omega, const double* __restrict__ Om_t,
               const double* __restrict__ Th_t, const double* __restrict__ X, const double* __restrict__ S,
               double lambda1, double lambda2, double sigma, int K, int p, double* __restrict__ Theta,
               double* __restrict__ G, unsigned char* __restrict__ code, double* __restrict__ jscale,
               double* __restrict__ partials, const double* flag)
{
    extern __shared__ double ysm[];                 // K * PD_PSLOT
    __shared__ double scratch[PD_NPART * 32];
    const int I = blockIdx.y, J = blockIdx.x, nt = gridDim.x;
    if (I > J) return;
    if (pd_done(flag)) return;
    const double l1 = sigma * lambda1, l2 = sigma * lambda2;
    const int tr = threadIdx.x / PD_PT, tc = threadIdx.x % PD_PT;
    const size_t pp = (size_t)p * p;
    const int i = I * PD_PT + tr, j = J * PD_PT + tc;
    const bool valid = (i < p) && (j < p);
    const bool upper = valid && (I < J || tr <= tc);
    const int slot = tr * PD_PLD + tc;
    double acc[PD_NPART] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};

    if (upper) {
        const size_t e = (size_t)i * p + j, et = (size_t)j * p + i;
        for (int k = 0; k < K; ++k) ysm[k * PD_PSLOT + slot] = V[k * pp + e];
        double* y = ysm + slot;
        if (i != j) {
            if (REG == 0) {
                double ss = 0.0;
                for (int k = 0; k < K; ++k) {
                    const double v = y[k * PD_PSLOT];
                    const unsigned char cd = fabs(v) > l1 ? 1 : 0;
                    code[k * pp + e] = cd; code[k * pp + et] = cd;
                    const double u = gg_soft(v, l1);
                    y[k * PD_PSLOT] = u;
                    ss += u * u;
                }
                const double nrm = sqrt(ss);
                const double a = nrm > l2 ? nrm : l2;
                const double f = a - l2;
                for (int k = 0; k < K; ++k) y[k * PD_PSLOT] = (y[k * PD_PSLOT] * f) / a;
                const double js = nrm > l2 ? l2 / nrm : -1.0;
                jscale[e] = js; jscale[et] = js;
            } else {
                gg_tv1d_inplace(y, K, PD_PSLOT, l2);
                long long prev = 0;
                for (int k = 0; k < K; ++k) {
                    const double z = y[k * PD_PSLOT];
                    const long long bits = __double_as_longlong(z);
                    const unsigned char cd = (fabs(z) > l1 ? 1 : 0) | ((k == 0 || bits != prev) ? 2 : 0);
                    code[k * pp + e] = cd; code[k * pp + et] = cd;
                    prev = bits;
                }
                for (int k = 0; k < K; ++k) y[k * PD_PSLOT] = gg_soft(y[k * PD_PSLOT], l1);
            }
            // P(Theta) on the strict upper triangle (ggl_helper.py:162-176), doubled at the end
            double n1 = 0.0, n2 = 0.0, prv = 0.0;
            for (int k = 0; k < K; ++k) {
                const double t = y[k * PD_PSLOT];
                n1 += fabs(t);
                if (REG == 0) n2 += t * t;
                else if (k > 0) n2 += fabs(t - prv);
                prv = t;
            }
            if (REG == 0) n2 = sqrt(n2);
            acc[1] += 2.0 * (lambda1 * n1 + lambda2 * n2);
        } else {
            for (int k = 0; k < K; ++k) code[k * pp + e] = 3;
        }
    }
    __syncthreads();

    const int sl0 = (I < J || tr <= tc) ? slot : (tc * PD_PLD + tr);
    const int i1 = J * PD_PT + tr, j1 = I * PD_PT + tc;          // element of the mirror tile (J,I)
    const bool ok1 = (I < J) && (i1 < p) && (j1 < p);
    const int sl1 = tc * PD_PLD + tr;
    for (int side = 0; side < 2; ++side) {
        const bool ok = side ? ok1 : valid;
        if (!ok) continue;
        const size_t e = side ? (size_t)i1 * p + j1 : (size_t)i * p + j;
        const int sl = side ? sl1 : sl0;
        for (int k = 0; k < K; ++k) {
            const size_t o = (size_t)k * pp + e;
            const double th = ysm[k * PD_PSLOT + sl];
            const double om = Omega[o], x = X[o];
            const double g = th - om;
            Theta[o] = th;
            G[o] = g;
            const double d3 = om - Om_t[o], d4 = th - Th_t[o];
            acc[0] += S[o] * om;
            acc[2] += x * (om - th);
            acc[3] += d3 * d3;
            acc[4] += d4 * d4;
            acc[5] += g * g;
        }
    }
    gg_block_sum<PD_NPART>(acc, scratch);
    if (threadIdx.x == 0) {
        double* out = partials + ((size_t)I * nt + J) * PD_NPART;
#pragma unroll
        for (int q = 0; q < PD_NPART; ++q) out[q] = acc[q];
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Out = sigma (Jphi + J_P[Din]) per entry (i,j) over the K instances; Jphi may be NULL (0) and may alias Out.
// partials (may be NULL): <Din, Out> per CTA.
template <int REG>
__global__ void __launch_bounds__(PD_THREADS)
pd_jp_kernel(const double* __restrict__ Din, const double* __restrict__ V, const unsigned char* __restrict__ code,
             const double* __restrict__ jscale, const double* Jphi, double sigma, double l1, int K, int p, double* Out,
             double* __restrict__ partials, const double* flag)
{
    __shared__ double scratch[32];
    if (pd_done(flag)) return;
    const size_t pp = (size_t)p * p;
    double acc[1] = {0.0};
    for (size_t e = (size_t)blockIdx.x * PD_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * PD_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        if (i == j) {
            for (int k = 0; k < K; ++k) {
                const size_t o = (size_t)k * pp + e;
                const double d = Din[o];
                const double out = sigma * ((Jphi ? Jphi[o] : 0.0) + d);
                Out[o] = out;
                acc[0] += d * out;
            }
        } else if (REG == 0) {
            const double sc = jscale[e];
            double ud = 0.0, uu = 0.0;
            if (sc >= 0.0) {
                for (int k = 0; k < K; ++k) {
                    const size_t o = (size_t)k * pp + e;
                    const double u = gg_soft(V[o], l1);
                    ud += u * Din[o];
                    uu += u * u;
                }
            }
            const double w = sc >= 0.0 ? ud / uu : 0.0;
            for (int k = 0; k < K; ++k) {
                const size_t o = (size_t)k * pp + e;
                const double d = Din[o];
                double jp = 0.0;
                if (sc >= 0.0) {
                    const double md = (code[o] & 1) ? d : 0.0;
                    jp = md - sc * (md - gg_soft(V[o], l1) * w);
                }
                const double out = sigma * ((Jphi ? Jphi[o] : 0.0) + jp);
                Out[o] = out;
                acc[0] += d * out;
            }
        } else {
            int k0 = 0;
            double sum = 0.0;
            for (int k = 0; k < K; ++k) {
                sum += Din[(size_t)k * pp + e];
                if (k == K - 1 || (code[(size_t)(k + 1) * pp + e] & 2)) {
                    const double avg = (code[(size_t)k * pp + e] & 1) ? sum / (double)(k - k0 + 1) : 0.0;
                    for (int kk = k0; kk <= k; ++kk) {
                        const size_t o = (size_t)kk * pp + e;
                        const double out = sigma * ((Jphi ? Jphi[o] : 0.0) + avg);
                        Out[o] = out;
                        acc[0] += Din[o] * out;
                    }
                    k0 = k + 1;
                    sum = 0.0;
                }
            }
        }
    }
    if (partials) {
        gg_block_sum<1>(acc, scratch);
        if (threadIdx.x == 0) partials[blockIdx.x] = acc[0];
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// CG on the device
__global__ void __launch_bounds__(PD_THREADS)
pd_cg_init_kernel(const double* __restrict__ G, size_t n, double* __restrict__ d, double* __restrict__ r,
                  double* __restrict__ pv, double* __restrict__ partials)
{
    __shared__ double scratch[32];
    double acc[1] = {0.0};
    for (size_t e = (size_t)blockIdx.x * PD_THREADS + threadIdx.x; e < n; e += (size_t)gridDim.x * PD_THREADS) {
        const double v = -G[e];
        d[e] = 0.0; r[e] = v; pv[e] = v;
        acc[0] += v * v;
    }
    gg_block_sum<1>(acc, scratch);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc[0];
}

// mode 0: init (|r|^2, tol^2, cap), 1: alpha = |r|^2 / <p,Hp>, 2: |r_new|^2, stop test, beta
__global__ void __launch_bounds__(PD_THREADS)
pd_cg_scalar_kernel(const double* __restrict__ partials, int nparts, int mode, double tol2, double cap, double* cg)
{
    __shared__ double scratch[32];
    if (mode != 0 && cg[CG_DONE] != 0.0) return;
    double acc[1] = {0.0};
    for (int t = threadIdx.x; t < nparts; t += PD_THREADS) acc[0] += partials[t];
    gg_block_sum<1>(acc, scratch);
    if (threadIdx.x != 0) return;
    const double s = acc[0];
    if (mode == 0) {
        cg[CG_RR] = s; cg[CG_TOL2] = tol2; cg[CG_CAP] = cap; cg[CG_ITER] = 0.0;
        cg[CG_ALPHA] = 0.0; cg[CG_BETA] = 0.0;
        cg[CG_DONE] = (s <= tol2 || cap <= 0.0 || !isfinite(s)) ? 1.0 : 0.0;
    } else if (mode == 1) {
        if (!(s > 0.0) || !isfinite(s)) { cg[CG_DONE] = 1.0; return; }
        cg[CG_ALPHA] = cg[CG_RR] / s;
    } else {
        const double it = cg[CG_ITER] + 1.0;
        cg[CG_ITER] = it;
        cg[CG_BETA] = s / cg[CG_RR];
        cg[CG_RR] = s;
        if (s <= cg[CG_TOL2] || it >= cg[CG_CAP] || !isfinite(s)) cg[CG_DONE] = 1.0;
    }
}

__global__ void __launch_bounds__(PD_THREADS)
pd_cg_update_kernel(const double* __restrict__ pv, const double* __restrict__ q, size_t n, double* __restrict__ d,
                    double* __restrict__ r, double* __restrict__ partials, const double* __restrict__ cg)
{
    __shared__ double scratch[32];
    if (cg[CG_DONE] != 0.0) return;
    const double a = cg[CG_ALPHA];
    double acc[1] = {0.0};
    for (size_t e = (size_t)blockIdx.x * PD_THREADS + threadIdx.x; e < n; e += (size_t)gridDim.x * PD_THREADS) {
        d[e] = d[e] + a * pv[e];
        const double rn = r[e] - a * q[e];
        r[e] = rn;
        acc[0] += rn * rn;
    }
    gg_block_sum<1>(acc, scratch);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc[0];
}

__global__ void __launch_bounds__(PD_THREADS)
pd_cg_p_kernel(const double* __restrict__ r, size_t n, double* __restrict__ pv, const double* __restrict__ cg)
{
    if (cg[CG_DONE] != 0.0) return;
    const double b = cg[CG_BETA];
    for (size_t e = (size_t)blockIdx.x * PD_THREADS + threadIdx.x; e < n; e += (size_t)gridDim.x * PD_THREADS)
        pv[e] = r[e] + b * pv[e];
}

// =====================================================================================================================
// host launchers (C++ linkage; the extern "C" ABI lives in gg_capi.cu)
// =====================================================================================================================
template <bool SYM, bool GAMMA>
static int launch_tn(const double* A, const double* fA, const double* B, int M, int p, double* C, const double* phi,
                     double sigma, const double* flag, cudaStream_t st)
{
    const int nt = (p + PD_TT - 1) / PD_TT;
    dim3 grid(nt, nt, M);
    gg_count_launch(1);
    if ((p & 1) == 0) pd_tn_kernel<SYM, GAMMA, true><<<grid, 256, 0, st>>>(A, fA, B, p, C, phi, sigma, flag);
    else pd_tn_kernel<SYM, GAMMA, false><<<grid, 256, 0, st>>>(A, fA, B, p, C, phi, sigma, flag);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_ppdna_build(const double* Om_t, const double* Th_t, const double* S, const double* X, const double* dX,
                          double s, double sigma, int K, int p, double* Xs, double* W, double* V, const double* flag,
                          cudaStream_t st)
{
    const size_t n = (size_t)K * p * p;
    gg_count_launch(1);
    pd_build_kernel<<<pd_blocks(n), PD_THREADS, 0, st>>>(Om_t, Th_t, S, X, dX, s, sigma, n, Xs, W, V, flag);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_ppdna_spectral(const double* Vt, const double* D, double sigma, int K, int p, double* Q, double* phi,
                             double* logdet, double* Omega, const double* flag, cudaStream_t st)
{
    gg_count_launch(2);
    pd_phi_kernel<<<K, PD_THREADS, 0, st>>>(D, sigma, p, phi, logdet, flag);
    GG_CHECK_LAUNCH();
    dim3 tg((p + 31) / 32, (p + 31) / 32, K);
    pd_transpose_kernel<<<tg, dim3(32, 8), 0, st>>>(Vt, p, Q, flag);
    GG_CHECK_LAUNCH();
    return launch_tn<true, false>(Vt, phi, Vt, K, p, Omega, nullptr, sigma, flag, st);
}

extern "C" int gg_ppdna_nparts(int p) { const int nt = (p + PD_PT - 1) / PD_PT; return nt * nt; }

int gg_launch_ppdna_prox(const double* V, const double* Omega, const double* Om_t, const double* Th_t, const double* X,
                         const double* S, double lambda1, double lambda2, double sigma, int reg, int K, int p,
                         double* Theta, double* G, unsigned char* code, double* jscale, double* partials,
                         const double* flag, cudaStream_t st)
{
    const int nt = (p + PD_PT - 1) / PD_PT;
    const size_t smem = (size_t)K * PD_PSLOT * sizeof(double);
    if (smem > 200 * 1024) return -2;   // K too large for the shared-memory layout
    auto kern = reg == 0 ? pd_prox_kernel<0> : pd_prox_kernel<1>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    gg_count_launch(1);
    kern<<<dim3(nt, nt), PD_PT * PD_PT, smem, st>>>(V, Omega, Om_t, Th_t, X, S, lambda1, lambda2, sigma, K, p, Theta,
                                                    G, code, jscale, partials, flag);
    GG_CHECK_LAUNCH();
    return 0;
}

extern "C" int gg_ppdna_jp_nparts(int p) { return pd_blocks((size_t)p * p); }

int gg_launch_ppdna_jp(const double* Din, const double* V, const unsigned char* code, const double* jscale,
                       const double* Jphi, double sigma, double lambda1, int reg, int K, int p, double* Out,
                       double* partials, const double* flag, cudaStream_t st)
{
    const int nb = pd_blocks((size_t)p * p);
    const double l1 = sigma * lambda1;
    gg_count_launch(1);
    if (reg == 0) pd_jp_kernel<0><<<nb, PD_THREADS, 0, st>>>(Din, V, code, jscale, Jphi, sigma, l1, K, p, Out, partials, flag);
    else pd_jp_kernel<1><<<nb, PD_THREADS, 0, st>>>(Din, V, code, jscale, Jphi, sigma, l1, K, p, Out, partials, flag);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_ppdna_hess(const double* Vt, const double* Q, const double* phi, const double* Din, const double* V,
                         const unsigned char* code, const double* jscale, double sigma, double lambda1, int reg, int K,
                         int p, double* Y, double* Z, double* Out, double* partials, const double* flag, cudaStream_t st)
{
    int rc;
    if ((rc = launch_tn<false, false>(Din, nullptr, Q, K, p, Y, nullptr, sigma, flag, st))) return rc;   // Y = D Q
    if ((rc = launch_tn<true, true>(Q, nullptr, Y, K, p, Z, phi, sigma, flag, st))) return rc;          // Z = Gamma o Q^T D Q
    if ((rc = launch_tn<false, false>(Z, nullptr, Vt, K, p, Y, nullptr, sigma, flag, st))) return rc;   // Y = Z Q^T
    if ((rc = launch_tn<true, false>(Vt, nullptr, Y, K, p, Out, nullptr, sigma, flag, st))) return rc;  // Out = Q Y
    return gg_launch_ppdna_jp(Din, V, code, jscale, Out, sigma, lambda1, reg, K, p, Out, partials, flag, st);
}

int gg_launch_ppdna_cg_init(const double* G, int K, int p, double tol, int max_iter, double* d, double* r, double* pv,
                            double* cg, double* partials, cudaStream_t st)
{
    const size_t n = (size_t)K * p * p;
    const int nb = pd_blocks(n);
    gg_count_launch(2);
    pd_cg_init_kernel<<<nb, PD_THREADS, 0, st>>>(G, n, d, r, pv, partials);
    GG_CHECK_LAUNCH();
    pd_cg_scalar_kernel<<<1, PD_THREADS, 0, st>>>(partials, nb, 0, tol * tol, (double)max_iter, cg);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_ppdna_cg(int iters, const double* Vt, const double* Q, const double* phi, const double* V,
                       const unsigned char* code, const double* jscale, double sigma, double lambda1, int reg, int K,
                       int p, double* d, double* r, double* pv, double* q, double* Y, double* Z, double* cg,
                       double* partials, cudaStream_t st)
{
    const size_t n = (size_t)K * p * p;
    const int nb = pd_blocks(n), njp = pd_blocks((size_t)p * p);
    const double* done = cg + CG_DONE;
    for (int it = 0; it < iters; ++it) {
        int rc = gg_launch_ppdna_hess(Vt, Q, phi, pv, V, code, jscale, sigma, lambda1, reg, K, p, Y, Z, q, partials,
                                      done, st);
        if (rc) return rc;
        gg_count_launch(4);
        pd_cg_scalar_kernel<<<1, PD_THREADS, 0, st>>>(partials, njp, 1, 0.0, 0.0, cg);
        GG_CHECK_LAUNCH();
        pd_cg_update_kernel<<<nb, PD_THREADS, 0, st>>>(pv, q, n, d, r, partials, cg);
        GG_CHECK_LAUNCH();
        pd_cg_scalar_kernel<<<1, PD_THREADS, 0, st>>>(partials, nb, 2, 0.0, 0.0, cg);
        GG_CHECK_LAUNCH();
        pd_cg_p_kernel<<<nb, PD_THREADS, 0, st>>>(r, n, pv, cg);
        GG_CHECK_LAUNCH();
    }
    return 0;
}
