// gg_jacobi.cu -- batched FP64 symmetric eigensolver for the Omega / L steps (sm_100a).
//
// Replaces the np.linalg.eigh call sites of the reference (admm_solver.py:181,199;
// single_admm_solver.py:164,174).  Only Q f(D) Q^T products are consumed downstream, so the
// solver returns eigenvectors as ROWS of Vt in arbitrary order with arbitrary signs.
//
// Method (one-sided Jacobi on an SPD-shifted matrix, "no-V" variant):
//   1. Gershgorin interval [lo,hi] of A  ->  sigma = 2h - c  (c centre, h half width), so that
//      A_s = A + sigma I has its spectrum inside [h, 3h]  (condition number <= 3).
//   2. Orthogonalise the rows of G = A_s by plane rotations (G <- J^T G).  At convergence
//      G = Lambda_s V^T, hence  lambda_i = |g_i| - sigma  and  v_i = g_i / |g_i|;
//      no separate eigenvector accumulation is needed, and because A_s is well conditioned the
//      Gram matrices used by the blocked variant lose no accuracy.
//   p <= GG_SMALL_MAX : whole matrix in shared memory, one CTA per matrix (jacobi_small_kernel).
//   larger p          : block one-sided Jacobi.  Per round-robin round one CTA per block pair (I,J):
//                       H = P P^T over the 2b rows of the pair on FP64 tensor cores (DMMA m8n8k4),
//                       eigenvectors U of H by the same shared-memory Jacobi, P <- U^T P by DMMA.
#include "gg_common.cuh"
#include "gg_jacobi_dev.cuh"
#include <stdlib.h>

#define GG_SMALL_MAX 160            // largest matrix the shared-memory Jacobi kernel can hold
#define GG_JACOBI_DEFAULT_MAX 48     // default crossover: above it the tridiagonal path is faster (p=100: 0.65 vs 1.86 ms)
#define JS_THREADS 1024
#define JS_LP 16

// ==========================================================================================
// small path: one CTA per matrix, everything in shared memory
// ==========================================================================================
// Vwarm (optional, (M,p,p), rows = orthonormal vectors): ADMM-aware warm start.  The iterates change slowly,
// so the previous iteration's eigenvectors nearly diagonalise the new matrix: starting the row
// orthogonalisation from G = Vwarm * A_s instead of A_s cuts the sweeps from ~9 to 2-4.  On exit Vwarm is
// overwritten by the new eigenvectors.
template <int NE>
__global__ void __launch_bounds__(JS_THREADS)
jacobi_small_kernel(double* __restrict__ A, double* __restrict__ D, int p, double tol, int max_sweeps,
                    const double* __restrict__ ctrl, int mpp, int* __restrict__ sweeps_out,
                    double* __restrict__ Vwarm)
{
    extern __shared__ double G[];            // p x ld
    __shared__ double red[64];
    __shared__ double s_sigma;
    const int m = blockIdx.x;
    if (ctrl && ctrl[(size_t)(m / mpp) * GG_CTRL_STRIDE + GG_C_DONE] != 0.0) return;
    const int ld = p | 1;
    double* Am = A + (size_t)m * p * p;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int e = threadIdx.x; e < p * p; e += blockDim.x) {
        const int i = e / p, jj = e - i * p;
        G[i * ld + jj] = Am[e];
    }
    __syncthreads();
    // Gershgorin bounds
    double lo = 1.0e300, hi = -1.0e300;
    for (int i = threadIdx.x; i < p; i += blockDim.x) {
        double rs = 0.0;
        for (int jj = 0; jj < p; ++jj) rs += fabs(G[i * ld + jj]);
        const double d = G[i * ld + i];
        rs -= fabs(d);
        lo = fmin(lo, d - rs);
        hi = fmax(hi, d + rs);
    }
    const double nlo = gg_block_max(-lo, red);
    __syncthreads();
    const double nhi = gg_block_max(hi, red + 32);
    if (threadIdx.x == 0) {
        const double l = -nlo, h2 = nhi;
        const double c = 0.5 * (l + h2);
        double h = 0.5 * (h2 - l);
        if (!(h > 0.0)) h = fmax(fabs(c), 1.0);
        s_sigma = 2.0 * h - c;
    }
    __syncthreads();
    const double sigma = s_sigma;
    if (Vwarm == nullptr) {
        for (int i = threadIdx.x; i < p; i += blockDim.x) G[i * ld + i] += sigma;
    } else {
        // G <- Vwarm * (A + sigma I); A is re-read from global/L1 (the shared copy is being overwritten)
        const double* Vw = Vwarm + (size_t)m * p * p;
        __syncthreads();
        for (int o = threadIdx.x; o < p * p; o += blockDim.x) {
            const int c = o / p, jj = o - c * p;
            const double* vr = Vw + (size_t)c * p;
            double acc = sigma * vr[jj];
#pragma unroll 4
            for (int k = 0; k < p; ++k) acc = fma(vr[k], Am[(size_t)k * p + jj], acc);
            G[c * ld + jj] = acc;
        }
    }
    __syncthreads();

    const int sw = jacobi_rows_smem<JS_LP, NE>(G, p, ld, tol, max_sweeps);
    if (threadIdx.x == 0 && sweeps_out) sweeps_out[m] = sw;
    __syncthreads();

    // finalise: lambda_i = |g_i| - sigma ; v_i = g_i / |g_i|
    double* Vw = Vwarm ? Vwarm + (size_t)m * p * p : nullptr;
    for (int i = wid; i < p; i += nw) {
        double ss = 0.0;
        for (int e = lane; e < p; e += 32) { const double x = G[i * ld + e]; ss = fma(x, x, ss); }
        ss = gg_warp_sum(ss);
        const double nrm = sqrt(ss);
        const double inv = 1.0 / nrm;
        if (lane == 0) D[(size_t)m * p + i] = nrm - sigma;
        for (int e = lane; e < p; e += 32) {
            const double v = G[i * ld + e] * inv;
            Am[(size_t)i * p + e] = v;
            if (Vw) Vw[(size_t)i * p + e] = v;
        }
    }
}

// ==========================================================================================
// block path
// ==========================================================================================
struct BjState {
    double* sigma;                 // (M)
    double* rowlo;                 // (M*p)
    double* rowhi;                 // (M*p)
    int* conv;                     // (M) 1 once matrix m has converged
    int* rotcount;                 // (M) block pairs updated in the current sweep
    unsigned long long* maxoff;    // (M) bit pattern of the largest off-measure seen in the sweep
    int* flags;                    // [0] = all matrices converged
};

__global__ void __launch_bounds__(256)
gersh_rows_kernel(const double* __restrict__ A, int p, double* __restrict__ rowlo, double* __restrict__ rowhi)
{
    const int m = blockIdx.y;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int i = blockIdx.x * 8 + wid;
    if (i >= p) return;
    const double* a = A + (size_t)m * p * p + (size_t)i * p;
    double rs = 0.0;
    for (int j = lane; j < p; j += 32)
        if (j != i) rs += fabs(a[j]);
    rs = gg_warp_sum(rs);
    if (lane == 0) {
        // The rounded sum can fall short of the exact off-diagonal sum by a relative (p-2)u, whatever the order;
        // widened by 2pu (u = 2^-53) it no longer can, so rowlo is a true lower bound of the row's disc and a
        // positive rowlo certifies positive definiteness.  (Summing |a_ii| into the row sum and subtracting it again
        // would let that sum's rounding turn an exact bound <= 0 into a positive one.)
        rs *= 1.0 + 2.0 * p * 1.1102230246251565e-16;
        const double d = a[i];
        rowlo[(size_t)m * p + i] = d - rs;
        rowhi[(size_t)m * p + i] = d + rs;
    }
}

__global__ void __launch_bounds__(256)
gersh_shift_kernel(double* __restrict__ A, int p, BjState st, const double* __restrict__ ctrl, int mpp)
{
    __shared__ double red[64];
    __shared__ double s_sigma;
    const int m = blockIdx.x;
    double lo = 1.0e300, hi = -1.0e300;
    for (int i = threadIdx.x; i < p; i += blockDim.x) {
        lo = fmin(lo, st.rowlo[(size_t)m * p + i]);
        hi = fmax(hi, st.rowhi[(size_t)m * p + i]);
    }
    const double nlo = gg_block_max(-lo, red);
    __syncthreads();
    const double nhi = gg_block_max(hi, red + 32);
    if (threadIdx.x == 0) {
        const double l = -nlo, h2 = nhi;
        const double c = 0.5 * (l + h2);
        double h = 0.5 * (h2 - l);
        if (!(h > 0.0)) h = fmax(fabs(c), 1.0);
        s_sigma = 2.0 * h - c;
        st.sigma[m] = s_sigma;
        const bool done = ctrl && ctrl[(size_t)(m / mpp) * GG_CTRL_STRIDE + GG_C_DONE] != 0.0;
        st.conv[m] = done ? 1 : 0;
        st.rotcount[m] = 0;
        st.maxoff[m] = 0ull;
        if (m == 0) st.flags[0] = 0;
    }
    __syncthreads();
    if (st.conv[m]) return;
    const double sigma = s_sigma;
    double* a = A + (size_t)m * p * p;
    for (int i = threadIdx.x; i < p; i += blockDim.x) a[(size_t)i * p + i] += sigma;
}

// One CTA per block pair.  NB2 = 2b rows per pair; KC = column chunk streamed through smem.
template <int NB2, int KC, bool VEC>
__global__ void __launch_bounds__(256)
bj_round_kernel(double* __restrict__ G, int p, int nb, int round, double tol, double tol_in, int inner_max_sweeps,
                BjState st)
{
    constexpr int B = NB2 / 2;
    constexpr int LDH = NB2 + 4;           // (4*row + col) mod 16 distinct for DMMA fragment loads
    constexpr int LDT = KC + 4;
    constexpr int NT = NB2 / 8;            // 8x8 DMMA tiles per side
    constexpr int WR = NT >= 8 ? 8 : NT;   // warps along tile rows
    constexpr int WC = 8 / WR;             // warps along tile cols
    constexpr int RPW = NT / WR;           // tile rows per warp
    constexpr int CPW = NT / WC;           // gram tile cols per warp
    constexpr int UT = KC / 8;             // update tile cols per chunk
    constexpr int UCPW = UT / WC;          // update tile cols per warp
    static_assert(UT % WC == 0 && UCPW >= 1, "tile split");

    extern __shared__ double smem[];
    double* Hs = smem;                                  // NB2 x LDH
    double* Ts = smem + NB2 * LDH;                      // 2 x NB2 x LDT
    __shared__ double red[32];
    __shared__ int s_skip;

    const int m = blockIdx.y;
    if (st.conv[m]) return;
    const int nbe = nb + (nb & 1);
    int I, J;
    rr_pair(nbe, round, blockIdx.x, I, J);
    if (I > J) { const int t = I; I = J; J = t; }
    if (J >= nb) return;

    double* Gm = G + (size_t)m * p * p;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;           // fragment row / col
    const int wr = wid / WC, wc = wid % WC;
    const int nchunks = (p + KC - 1) / KC;

    auto grow = [&](int t) -> int { return t < B ? I * B + t : J * B + (t - B); };

    auto load_chunk = [&](int c, int buf) {
        double* T = Ts + (size_t)buf * NB2 * LDT;
        const int k0 = c * KC;
        if (VEC) {
            for (int idx = tid; idx < NB2 * (KC / 2); idx += 256) {
                const int t = idx / (KC / 2), kk = (idx % (KC / 2)) * 2;
                const int gr = grow(t), gc = k0 + kk;
                double* dst = T + t * LDT + kk;
                if (gr < p && gc < p) gg_cp_async16(dst, Gm + (size_t)gr * p + gc);   // p even: gc+1 < p too
                else { dst[0] = 0.0; dst[1] = 0.0; }
            }
        } else {
            for (int idx = tid; idx < NB2 * KC; idx += 256) {
                const int t = idx / KC, kk = idx % KC;
                const int gr = grow(t), gc = k0 + kk;
                double* dst = T + t * LDT + kk;
                if (gr < p && gc < p) gg_cp_async8(dst, Gm + (size_t)gr * p + gc);
                else dst[0] = 0.0;
            }
        }
        gg_cp_commit();
    };

    // ---------------- phase 1: H = P P^T ---------------------------------------------------
    double acc[RPW][CPW][2];
#pragma unroll
    for (int a = 0; a < RPW; ++a)
#pragma unroll
        for (int b = 0; b < CPW; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }

    load_chunk(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) { load_chunk(c + 1, (c + 1) & 1); gg_cp_wait<1>(); }
        else gg_cp_wait<0>();
        __syncthreads();
        const double* T = Ts + (size_t)(c & 1) * NB2 * LDT;
#pragma unroll
        for (int k0 = 0; k0 < KC; k0 += 4) {
            double fa[RPW], fb[CPW];
#pragma unroll
            for (int a = 0; a < RPW; ++a) fa[a] = T[((wr * RPW + a) * 8 + fr) * LDT + k0 + fc];
#pragma unroll
            for (int b = 0; b < CPW; ++b) fb[b] = T[((wc * CPW + b) * 8 + fr) * LDT + k0 + fc];
#pragma unroll
            for (int a = 0; a < RPW; ++a)
#pragma unroll
                for (int b = 0; b < CPW; ++b) gg_dmma(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < RPW; ++a)
#pragma unroll
        for (int b = 0; b < CPW; ++b) {
            const int r = (wr * RPW + a) * 8 + fr, cc = (wc * CPW + b) * 8 + 2 * fc;
            Hs[r * LDH + cc] = acc[a][b][0];
            Hs[r * LDH + cc + 1] = acc[a][b][1];
        }
    __syncthreads();

    // ---------------- phase 2: convergence measure, inner eigenproblem ----------------------
    double mx = 0.0;
    for (int idx = tid; idx < NB2 * NB2; idx += 256) {
        const int i = idx / NB2, j = idx % NB2;
        if (j > i) {
            const double dd = Hs[i * LDH + i] * Hs[j * LDH + j];
            if (dd > 0.0) mx = fmax(mx, fabs(Hs[i * LDH + j]) / sqrt(dd));
        }
    }
    mx = gg_block_max(mx, red);
    if (tid == 0) {
        s_skip = (mx <= tol) ? 1 : 0;
        atomicMax(st.maxoff + m, (unsigned long long)__double_as_longlong(mx));
        if (mx > tol) atomicAdd(st.rotcount + m, 1);
    }
    __syncthreads();
    if (s_skip) return;

    jacobi_rows_smem<8, NB2 / 8>(Hs, NB2, LDH, tol_in, inner_max_sweeps);
    __syncthreads();
    // rows of Hs are now sigma_i * u_i ; normalise -> Ut (row i = eigenvector i). Zero rows -> e_i.
    for (int i = wid; i < NB2; i += 8) {
        double ss = 0.0;
        for (int e = lane; e < NB2; e += 32) { const double x = Hs[i * LDH + e]; ss = fma(x, x, ss); }
        ss = gg_warp_sum(ss);
        if (ss > 0.0) {
            const double inv = rsqrt(ss);
            for (int e = lane; e < NB2; e += 32) Hs[i * LDH + e] *= inv;
        } else {
            for (int e = lane; e < NB2; e += 32) Hs[i * LDH + e] = (e == i) ? 1.0 : 0.0;
        }
    }
    __syncthreads();

    // ---------------- phase 3: P <- Ut * P  (in place, chunk by chunk) -----------------------
    load_chunk(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) { load_chunk(c + 1, (c + 1) & 1); gg_cp_wait<1>(); }
        else gg_cp_wait<0>();
        __syncthreads();
        const double* T = Ts + (size_t)(c & 1) * NB2 * LDT;
        double o[RPW][UCPW][2];
#pragma unroll
        for (int a = 0; a < RPW; ++a)
#pragma unroll
            for (int b = 0; b < UCPW; ++b) { o[a][b][0] = 0.0; o[a][b][1] = 0.0; }
#pragma unroll 4
        for (int m0 = 0; m0 < NB2; m0 += 4) {
            double fa[RPW], fb[UCPW];
#pragma unroll
            for (int a = 0; a < RPW; ++a) fa[a] = Hs[((wr * RPW + a) * 8 + fr) * LDH + m0 + fc];
#pragma unroll
            for (int b = 0; b < UCPW; ++b) fb[b] = T[(m0 + fc) * LDT + (wc * UCPW + b) * 8 + fr];
#pragma unroll
            for (int a = 0; a < RPW; ++a)
#pragma unroll
                for (int b = 0; b < UCPW; ++b) gg_dmma(o[a][b][0], o[a][b][1], fa[a], fb[b]);
        }
        const int k0 = c * KC;
#pragma unroll
        for (int a = 0; a < RPW; ++a) {
            const int gr = grow((wr * RPW + a) * 8 + fr);
            if (gr < p) {
#pragma unroll
                for (int b = 0; b < UCPW; ++b) {
                    const int gc = k0 + (wc * UCPW + b) * 8 + 2 * fc;
                    double* dst = Gm + (size_t)gr * p + gc;
                    if (VEC) {
                        if (gc < p) *reinterpret_cast<double2*>(dst) = make_double2(o[a][b][0], o[a][b][1]);
                    } else {
                        if (gc < p) dst[0] = o[a][b][0];
                        if (gc + 1 < p) dst[1] = o[a][b][1];
                    }
                }
            }
        }
        __syncthreads();
    }
}

__global__ void bj_sweep_end_kernel(BjState st, int M, double quad_tol)
{
    __shared__ int s_all;
    if (threadIdx.x == 0) s_all = 1;
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        if (!st.conv[m]) {
            const double mo = __longlong_as_double((long long)st.maxoff[m]);
            if (st.rotcount[m] == 0 || mo < quad_tol) st.conv[m] = 1;
            else atomicAnd(&s_all, 0);
        }
        st.rotcount[m] = 0;
        st.maxoff[m] = 0ull;
    }
    __syncthreads();
    if (threadIdx.x == 0) st.flags[0] = s_all;
}

__global__ void __launch_bounds__(256)
bj_finalize_kernel(double* __restrict__ G, double* __restrict__ D, int p, BjState st,
                   const double* __restrict__ ctrl, int mpp, int normalize)
{
    const int m = blockIdx.y;
    if (ctrl && ctrl[(size_t)(m / mpp) * GG_CTRL_STRIDE + GG_C_DONE] != 0.0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int i = blockIdx.x * 8 + wid;
    if (i >= p) return;
    double* g = G + (size_t)m * p * p + (size_t)i * p;
    double ss = 0.0;
    for (int e = lane; e < p; e += 32) { const double x = g[e]; ss = fma(x, x, ss); }
    ss = gg_warp_sum(ss);
    const double nrm = sqrt(ss);
    if (lane == 0) D[(size_t)m * p + i] = nrm - st.sigma[m];
    if (normalize) {
        const double inv = 1.0 / nrm;
        for (int e = lane; e < p; e += 32) g[e] *= inv;
    }
}

// ==========================================================================================
// host side
// ==========================================================================================
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// matrices up to this size use the shared-memory Jacobi kernel (env GG_JACOBI_MAX, read once); it reads the FULL matrix,
// the tridiagonal path above it only the upper triangle -- the host loop asks for this value (gg_jacobi_max)
int gg_jacobi_small_max()
{
    static int small_max = -1;
    if (small_max < 0) {
        const char* ev = getenv("GG_JACOBI_MAX");
        int v = ev ? atoi(ev) : GG_JACOBI_DEFAULT_MAX;
        if (v > GG_SMALL_MAX) v = GG_SMALL_MAX;
        if (v < 32) v = 32;          // the D&C leaves need n > 32
        small_max = v;
    }
    return small_max;
}

size_t gg_tridiag_ws_bytes(int M, int n);
int gg_eigh_tridiag_impl(double* A, double* D, int M, int n, const double* ctrl, int mpp, void* wsp, size_t ws_bytes,
                         cudaStream_t s, int which);

static size_t gg_jacobi_ws_bytes(int M, int p)
{
    size_t b = 0;
    b += align_up(sizeof(double) * (size_t)M, 256);              // sigma
    b += 2 * align_up(sizeof(double) * (size_t)M * p, 256);      // rowlo, rowhi
    b += 2 * align_up(sizeof(int) * (size_t)M, 256);             // conv, rotcount
    b += align_up(sizeof(unsigned long long) * (size_t)M, 256);  // maxoff
    b += 256;                                                    // flags
    b += align_up(sizeof(int) * (size_t)M, 256);                 // sweeps (small path)
    return b;
}

size_t gg_eigh_ws_bytes(int M, int p)
{
    const size_t a = gg_jacobi_ws_bytes(M, p);
    const size_t b = (p > 32) ? gg_tridiag_ws_bytes(M, p) : 0;
    return a > b ? a : b;
}

template <int NB2, int KC>
static int launch_round(double* G, int M, int p, int nb, int round, double tol, double tol_in, int inner_max,
                        BjState st, cudaStream_t s)
{
    const size_t smem = sizeof(double) * ((size_t)NB2 * (NB2 + 4) + 2 * (size_t)NB2 * (KC + 4));
    const int nbe = nb + (nb & 1);
    dim3 grid(nbe / 2, M);
    if ((p & 1) == 0) {
        auto k = bj_round_kernel<NB2, KC, true>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   // per device: set on every call
        gg_count_launch(1);
        k<<<grid, 256, smem, s>>>(G, p, nb, round, tol, tol_in, inner_max, st);
    } else {
        auto k = bj_round_kernel<NB2, KC, false>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   // per device: set on every call
        gg_count_launch(1);
        k<<<grid, 256, smem, s>>>(G, p, nb, round, tol, tol_in, inner_max, st);
    }
    GG_CHECK_LAUNCH();
    return 0;
}

// A: (M,p,p) symmetric, overwritten by Vt (rows = eigenvectors, unit norm if `vectors`).
// D: (M,p) eigenvalues (unsorted).  info[0] = sweeps used (block path), 0 (small path: the per-matrix sweep counts
// stay on the device, in the last slot of the workspace), -1 (tridiagonal path).
int gg_eigh_impl(double* A, double* D, int M, int p, const double* ctrl, int mpp, void* ws, size_t ws_bytes,
                 int vectors, int block_nb2, double tol, int max_sweeps, double quad_tol, int* info,
                 double* Vwarm, cudaStream_t s)
{
    if (M <= 0 || p <= 0) return 0;
    if (ws_bytes < gg_jacobi_ws_bytes(M, p)) return -3;
    char* w = (char*)ws;
    BjState st;
    st.sigma = (double*)w; w += align_up(sizeof(double) * (size_t)M, 256);
    st.rowlo = (double*)w; w += align_up(sizeof(double) * (size_t)M * p, 256);
    st.rowhi = (double*)w; w += align_up(sizeof(double) * (size_t)M * p, 256);
    st.conv = (int*)w; w += align_up(sizeof(int) * (size_t)M, 256);
    st.rotcount = (int*)w; w += align_up(sizeof(int) * (size_t)M, 256);
    st.maxoff = (unsigned long long*)w; w += align_up(sizeof(unsigned long long) * (size_t)M, 256);
    st.flags = (int*)w; w += 256;
    int* sweeps_small = (int*)w;

    if (tol <= 0.0) tol = fmax(1.0e-14, 8.0 * 2.220446049250313e-16 * sqrt((double)p));
    if (max_sweeps <= 0) max_sweeps = 30;

    const int small_max = gg_jacobi_small_max();
    if (p <= small_max || (block_nb2 == 1 && p <= GG_SMALL_MAX)) {       // block_nb2 == 1 forces this path
        const int ld = p | 1;
        const size_t smem = sizeof(double) * (size_t)p * ld;
        const int maxsm = (int)(sizeof(double) * GG_SMALL_MAX * (GG_SMALL_MAX | 1));
        {   // the attribute is per device and cheap to set: no process-wide "done" flag
            cudaFuncSetAttribute(jacobi_small_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
            cudaFuncSetAttribute(jacobi_small_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
            cudaFuncSetAttribute(jacobi_small_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
            cudaFuncSetAttribute(jacobi_small_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
            cudaError_t e = cudaFuncSetAttribute(jacobi_small_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
            if (e != cudaSuccess) return (int)e;
        }
        // threads: 16 lanes per row pair; no more groups than pairs (rounded up to a warp multiple)
        int threads = ((p + 1) / 2) * JS_LP;
        threads = (threads + 31) / 32 * 32;
        if (threads > JS_THREADS) threads = JS_THREADS;
        if (threads < 64) threads = 64;
        const int ne = (p + JS_LP - 1) / JS_LP;
        gg_count_launch(1);
        if (ne <= 2) jacobi_small_kernel<2><<<M, threads, smem, s>>>(A, D, p, tol, max_sweeps, ctrl, mpp, sweeps_small, Vwarm);
        else if (ne <= 4) jacobi_small_kernel<4><<<M, threads, smem, s>>>(A, D, p, tol, max_sweeps, ctrl, mpp, sweeps_small, Vwarm);
        else if (ne <= 6) jacobi_small_kernel<6><<<M, threads, smem, s>>>(A, D, p, tol, max_sweeps, ctrl, mpp, sweeps_small, Vwarm);
        else if (ne <= 8) jacobi_small_kernel<8><<<M, threads, smem, s>>>(A, D, p, tol, max_sweeps, ctrl, mpp, sweeps_small, Vwarm);
        else jacobi_small_kernel<10><<<M, threads, smem, s>>>(A, D, p, tol, max_sweeps, ctrl, mpp, sweeps_small, Vwarm);
        GG_CHECK_LAUNCH();
        if (info) info[0] = 0;
        return 0;
    }

    // ---- large p: tridiagonalisation + divide & conquer (default), or block Jacobi on request ----
    if (block_nb2 != 32 && block_nb2 != 64 && block_nb2 != 128 && p > 7000) block_nb2 = 64;   // D&C smem limit
    if (block_nb2 != 32 && block_nb2 != 64 && block_nb2 != 128) {
        const int rc = gg_eigh_tridiag_impl(A, D, M, p, ctrl, mpp, ws, ws_bytes, s, vectors ? 0 : 4);
        if (info) info[0] = -1;
        return rc;
    }
    int nb2 = block_nb2;
    const int b = nb2 / 2;
    const int nb = (p + b - 1) / b;
    const int nbe = nb + (nb & 1);
    const double tol_in = 1.0e-15;

    dim3 grows((p + 7) / 8, M);
    gg_count_launch(1);
    gersh_rows_kernel<<<grows, 256, 0, s>>>(A, p, st.rowlo, st.rowhi);
    GG_CHECK_LAUNCH();
    gg_count_launch(1);
    gersh_shift_kernel<<<M, 256, 0, s>>>(A, p, st, ctrl, mpp);
    GG_CHECK_LAUNCH();

    int used = 0;
    for (int sweep = 0; sweep < max_sweeps; ++sweep) {
        for (int r = 0; r < nbe - 1; ++r) {
            int rc;
            if (nb2 == 32) rc = launch_round<32, 32>(A, M, p, nb, r, tol, tol_in, 30, st, s);
            else if (nb2 == 64) rc = launch_round<64, 32>(A, M, p, nb, r, tol, tol_in, 30, st, s);
            else rc = launch_round<128, 16>(A, M, p, nb, r, tol, tol_in, 30, st, s);
            if (rc) return rc;
        }
        gg_count_launch(1);
        bj_sweep_end_kernel<<<1, 256, 0, s>>>(st, M, quad_tol);
        GG_CHECK_LAUNCH();
        used = sweep + 1;
        if (sweep >= 1) {
            int h_flag = 0;
            cudaError_t e = cudaMemcpyAsync(&h_flag, st.flags, sizeof(int), cudaMemcpyDeviceToHost, s);
            if (e != cudaSuccess) return (int)e;
            e = cudaStreamSynchronize(s);
            if (e != cudaSuccess) return (int)e;
            if (h_flag) break;
        }
    }
    gg_count_launch(1);
    bj_finalize_kernel<<<grows, 256, 0, s>>>(A, D, p, st, ctrl, mpp, vectors);
    GG_CHECK_LAUNCH();
    if (info) info[0] = used;
    return 0;
}

// Gershgorin lower bound of the spectrum per matrix: out[m] = min_i (a_ii - sum_{j != i} |a_ij|).
// A positive value proves positive definiteness, so the post-loop PD check (admm_solver.py:294-296) can skip
// its eigendecomposition.
__global__ void __launch_bounds__(256)
gersh_min_kernel(const double* __restrict__ rowlo, int p, double* __restrict__ out)
{
    __shared__ double red[32];
    const int m = blockIdx.x;
    double lo = 1.0e300;
    for (int i = threadIdx.x; i < p; i += blockDim.x) lo = fmin(lo, rowlo[(size_t)m * p + i]);
    const double nlo = gg_block_max(-lo, red);
    if (threadIdx.x == 0) out[m] = -nlo;
}

int gg_gershgorin_min_impl(const double* A, int M, int p, void* ws, size_t ws_bytes, double* out, cudaStream_t s)
{
    if (ws_bytes < 2 * align_up(sizeof(double) * (size_t)M * p, 256)) return -3;
    double* rowlo = (double*)ws;
    double* rowhi = (double*)((char*)ws + align_up(sizeof(double) * (size_t)M * p, 256));
    dim3 grows((p + 7) / 8, M);
    gg_count_launch(1);
    gersh_rows_kernel<<<grows, 256, 0, s>>>(A, p, rowlo, rowhi);
    GG_CHECK_LAUNCH();
    gg_count_launch(1);
    gersh_min_kernel<<<M, 256, 0, s>>>(rowlo, p, out);
    GG_CHECK_LAUNCH();
    return 0;
}
