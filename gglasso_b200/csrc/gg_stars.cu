// gg_stars.cu -- device work of stability selection (StARS, Liu, Roeder & Wasserman 2010) (sm_100a).
//
// The data of all classes stay resident as one (sum n_k, p) FP64 array, class k starting at row rowoff[k].  A chunk
// of nsub subsamples is described by idx: for subsample s and class k the b_k row indices (within class k) at
// idx[s * bsum + boff[k] ..], bsum = boff[K].
//
//   gg_subsample_cov     S[s,k] = (1/b_k) Xc^T Xc over the rows idx[s,k,:] of class k, centred on their mean
//                        (np.cov(X_sub, rowvar=False, bias=True)), optionally scaled to S_ij / (sqrt(S_ii) sqrt(S_jj))
//   gg_edge_count        counts[l,k,i,j] += sum_s 1[Theta_{(s L + l) K + k}[i][j] != 0], i < j
//   gg_stars_instability per (l,k): sum_{i<j} 2 theta (1 - theta) / C(p,2) and sum_{i<j} count / B, theta = count / B
//
// Compiled with -fmad=false: the centring, the 1/b factor and the scaling are the separate roundings numpy performs.
#include "gg_common.cuh"

#define ST_THREADS 256
#define ST_TT 64               // output tile of the covariance product
#define ST_KC 16               // rows of the subsample per reduction chunk
#define ST_LD (ST_TT + 4)      // conflict-free fragment loads (as pd_tn_kernel)
#define ST_MEAN_COLS 128

// ---------------------------------------------------------------------------------------------------------------------
// Column means of every (s,k): one thread per column, rows summed in index order.  A column whose sampled values are all
// equal has zero variance; its index is folded into zero_col[s*K+k] with atomicMin (order-independent result).
__global__ void __launch_bounds__(ST_MEAN_COLS)
st_mean_kernel(const double* __restrict__ X, const int* __restrict__ rowoff, const int* __restrict__ idx,
               const int* __restrict__ boff, int K, int p, double* __restrict__ mean, int* __restrict__ zero_col)
{
    __shared__ int zmin;
    const int sk = blockIdx.y, s = sk / K, k = sk - s * K;
    const int j = blockIdx.x * ST_MEAN_COLS + threadIdx.x;
    if (threadIdx.x == 0) zmin = p;
    __syncthreads();
    if (j < p) {
        const int b = boff[k + 1] - boff[k];
        const int* ix = idx + (size_t)s * boff[K] + boff[k];
        const double* Xk = X + (size_t)rowoff[k] * p + j;
        const double x0 = Xk[(size_t)ix[0] * p];
        double sum = 0.0;
        bool flat = true;
        for (int r = 0; r < b; ++r) {
            const double x = Xk[(size_t)ix[r] * p];
            sum += x;
            flat = flat && (x == x0);
        }
        mean[(size_t)sk * p + j] = sum / (double)b;
        if (flat) atomicMin(&zmin, j);
    }
    __syncthreads();
    if (threadIdx.x == 0 && zmin < p) atomicMin(zero_col + sk, zmin);
}

// ---------------------------------------------------------------------------------------------------------------------
// S[sk] = (1/b) Xc^T Xc on DMMA m8n8k4: pd_tn_kernel's tile and warp shapes (64 x 64 per CTA, 16 x 32 per warp,
// cp.async double buffer), with the subsample's rows as the inner dimension.  Operand rows are gathered through idx;
// rows past b (and columns past p) are filled with the column mean (zero), so centring in the fragment load makes them
// exact zeros.  Only tiles I <= J are computed and the mirror tile is written through shared memory: S is exactly
// symmetric.
template <bool VEC>
__global__ void __launch_bounds__(ST_THREADS)
st_cov_kernel(const double* __restrict__ X, const int* __restrict__ rowoff, const int* __restrict__ idx,
              const int* __restrict__ boff, int K, int p, const double* __restrict__ mean, double* __restrict__ S)
{
    __shared__ __align__(16) double sm[2 * 2 * ST_KC * ST_LD];   // As[2][KC][LD], Bs[2][KC][LD]; reused as Cs[64][65]
    __shared__ double mus[2][ST_TT];
    const int I = blockIdx.y, J = blockIdx.x, sk = blockIdx.z;
    if (I > J) return;
    const int s = sk / K, k = sk - s * K;
    const int b = boff[k + 1] - boff[k];
    const int* ix = idx + (size_t)s * boff[K] + boff[k];
    const double* Xk = X + (size_t)rowoff[k] * p;
    const double* mu = mean + (size_t)sk * p;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;
    const int wr = wid >> 1, wc = wid & 1;
    const int i0 = I * ST_TT, j0 = J * ST_TT;
    const int nchunks = (b + ST_KC - 1) / ST_KC;

    if (tid < 2 * ST_TT) {
        const int which = tid / ST_TT, e = tid % ST_TT, g = (which ? j0 : i0) + e;
        mus[which][e] = g < p ? mu[g] : 0.0;
    }
    __syncthreads();

    auto load_chunk = [&](int c, int buf) {
        double* As = sm + (size_t)buf * ST_KC * ST_LD;
        double* Bs = sm + (size_t)(2 + buf) * ST_KC * ST_LD;
        const int c0 = c * ST_KC;
        if (VEC) {
            for (int t = tid; t < 2 * ST_KC * (ST_TT / 2); t += ST_THREADS) {
                const int which = t / (ST_KC * (ST_TT / 2));
                const int rem = t % (ST_KC * (ST_TT / 2));
                const int kk = rem / (ST_TT / 2), e = (rem % (ST_TT / 2)) * 2;
                const int gc = (which ? j0 : i0) + e, gr = c0 + kk;
                double* dst = (which ? Bs : As) + kk * ST_LD + e;
                if (gr < b && gc < p) gg_cp_async16(dst, Xk + (size_t)ix[gr] * p + gc);
                else { dst[0] = mus[which][e]; dst[1] = mus[which][e + 1]; }
            }
        } else {
            for (int t = tid; t < 2 * ST_KC * ST_TT; t += ST_THREADS) {
                const int which = t / (ST_KC * ST_TT);
                const int rem = t % (ST_KC * ST_TT);
                const int kk = rem / ST_TT, e = rem % ST_TT;
                const int gc = (which ? j0 : i0) + e, gr = c0 + kk;
                double* dst = (which ? Bs : As) + kk * ST_LD + e;
                if (gr < b && gc < p) gg_cp_async8(dst, Xk + (size_t)ix[gr] * p + gc);
                else dst[0] = mus[which][e];
            }
        }
        gg_cp_commit();
    };

    double ma[2], mb[4];
#pragma unroll
    for (int a = 0; a < 2; ++a) ma[a] = mus[0][(wr * 2 + a) * 8 + fr];
#pragma unroll
    for (int q = 0; q < 4; ++q) mb[q] = mus[1][(wc * 4 + q) * 8 + fr];

    double acc[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int q = 0; q < 4; ++q) { acc[a][q][0] = 0.0; acc[a][q][1] = 0.0; }

    load_chunk(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) { load_chunk(c + 1, (c + 1) & 1); gg_cp_wait<1>(); }
        else gg_cp_wait<0>();
        __syncthreads();
        const int buf = c & 1;
        const double* As = sm + (size_t)buf * ST_KC * ST_LD;
        const double* Bs = sm + (size_t)(2 + buf) * ST_KC * ST_LD;
#pragma unroll
        for (int k0 = 0; k0 < ST_KC; k0 += 4) {
            double fa[2], fb[4];
#pragma unroll
            for (int a = 0; a < 2; ++a) fa[a] = As[(k0 + fc) * ST_LD + (wr * 2 + a) * 8 + fr] - ma[a];
#pragma unroll
            for (int q = 0; q < 4; ++q) fb[q] = Bs[(k0 + fc) * ST_LD + (wc * 4 + q) * 8 + fr] - mb[q];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int q = 0; q < 4; ++q) gg_dmma(acc[a][q][0], acc[a][q][1], fa[a], fb[q]);
        }
        __syncthreads();
    }

    double* Cs = sm;                         // 64 x 65
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = (wr * 2 + a) * 8 + fr, cc = (wc * 4 + q) * 8 + 2 * fc;
            Cs[r * 65 + cc] = acc[a][q][0];
            Cs[r * 65 + cc + 1] = acc[a][q][1];
        }
    __syncthreads();
    const double inv_b = 1.0 / (double)b;    // numpy: c *= 1 / fact
    double* O = S + (size_t)sk * p * p;
    for (int t = tid; t < ST_TT * ST_TT; t += ST_THREADS) {
        const int r = t / ST_TT, cc = t % ST_TT;
        const int gi = i0 + r, gj = j0 + cc;
        if (gi < p && gj < p) O[(size_t)gi * p + gj] = ((I == J && cc < r) ? Cs[cc * 65 + r] : Cs[r * 65 + cc]) * inv_b;
    }
    if (I < J) {
        for (int t = tid; t < ST_TT * ST_TT; t += ST_THREADS) {
            const int r = t / ST_TT, cc = t % ST_TT;        // element (j0 + r, i0 + cc) of the mirror tile
            const int gi = j0 + r, gj = i0 + cc;
            if (gi < p && gj < p) O[(size_t)gi * p + gj] = Cs[cc * 65 + r] * inv_b;
        }
    }
}

// sq[sk][i] = sqrt(S[sk][i][i])  (the diagonal is read before st_scale_kernel overwrites it)
__global__ void __launch_bounds__(ST_THREADS)
st_diag_kernel(const double* __restrict__ S, int nmat, int p, double* __restrict__ sq)
{
    const size_t n = (size_t)nmat * p;
    for (size_t e = (size_t)blockIdx.x * ST_THREADS + threadIdx.x; e < n; e += (size_t)gridDim.x * ST_THREADS) {
        const size_t m = e / p, i = e - m * p;
        sq[e] = sqrt(S[(m * p + i) * p + i]);
    }
}

// S_ij / (sqrt(S_ii) sqrt(S_jj)), the expression of the reference's scale_array_by_diagonal (exactly symmetric)
__global__ void __launch_bounds__(ST_THREADS)
st_scale_kernel(double* __restrict__ S, int p, const double* __restrict__ sq)
{
    const size_t pp = (size_t)p * p, base = (size_t)blockIdx.y * pp;
    const double* d = sq + (size_t)blockIdx.y * p;
    for (size_t e = (size_t)blockIdx.x * ST_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * ST_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        S[base + e] = S[base + e] / (d[i] * d[j]);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// counts[l,k,i,j] += number of s < nsub with Theta[(s*L + l)*K + k][i][j] != 0, for i < j.  One thread per entry loops
// over s: no atomics, deterministic.  Entries i >= j of counts are not touched.
__global__ void __launch_bounds__(ST_THREADS)
st_edge_count_kernel(const double* __restrict__ Theta, int nsub, int L, int K, int p, int* __restrict__ counts)
{
    const size_t pp = (size_t)p * p;
    const int lk = blockIdx.y;                      // l * K + k
    const size_t step = (size_t)L * K * pp;         // from subsample s to s + 1
    for (size_t e = (size_t)blockIdx.x * ST_THREADS + threadIdx.x; e < pp; e += (size_t)gridDim.x * ST_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        if (i >= j) continue;
        const double* t = Theta + (size_t)lk * pp + e;
        int n = 0;
        for (int s = 0; s < nsub; ++s) n += (t[(size_t)s * step] != 0.0) ? 1 : 0;
        counts[(size_t)lk * pp + e] += n;
    }
}

// per (l,k), one CTA: the integer sums sum_{i<j} c (B - c) and sum_{i<j} c (exact, so independent of the order of
// the reduction), then out[lk][0] = 2 sum c (B - c) / (B^2 C(p,2)) and out[lk][1] = sum c / B.
__global__ void __launch_bounds__(ST_THREADS)
st_instability_kernel(const int* __restrict__ counts, int p, int B, double* __restrict__ out)
{
    __shared__ long long red[2][ST_THREADS / 32];
    const size_t pp = (size_t)p * p;
    const int* c = counts + (size_t)blockIdx.x * pp;
    long long v = 0, e1 = 0;
    for (size_t e = threadIdx.x; e < pp; e += ST_THREADS) {
        const int i = (int)(e / p), j = (int)(e - (size_t)i * p);
        if (i >= j) continue;
        const long long n = c[e];
        v += n * (B - n);
        e1 += n;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v += __shfl_xor_sync(0xffffffffu, v, o);
        e1 += __shfl_xor_sync(0xffffffffu, e1, o);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { red[0][wid] = v; red[1][wid] = e1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long sv = 0, se = 0;
        for (int w = 0; w < ST_THREADS / 32; ++w) { sv += red[0][w]; se += red[1][w]; }
        const double npairs = 0.5 * (double)p * (double)(p - 1);
        out[2 * (size_t)blockIdx.x] = (2.0 * (double)sv) / ((double)B * (double)B) / npairs;
        out[2 * (size_t)blockIdx.x + 1] = (double)se / (double)B;
    }
}

// =====================================================================================================================
// host launchers (C++ linkage; the extern "C" ABI lives in gg_capi.cu)
// =====================================================================================================================
static inline int st_blocks(size_t n, int per)
{
    size_t b = (n + ST_THREADS - 1) / ST_THREADS;
    const size_t cap = (size_t)(148 * 8 + per - 1) / per;
    if (b > cap) b = cap;
    return (int)(b < 1 ? 1 : b);
}

int gg_launch_subsample_cov(const double* X, const int* rowoff, const int* idx, const int* boff, int nsub, int K, int p,
                            int scale, double* mean, double* S, int* zero_col, cudaStream_t st)
{
    const int nmat = nsub * K;
    cudaError_t e = cudaMemsetAsync(zero_col, 0x7f, sizeof(int) * (size_t)nmat, st);   // 0x7f7f7f7f >= p: none yet
    if (e != cudaSuccess) return (int)e;
    gg_count_launch(1);
    st_mean_kernel<<<dim3((p + ST_MEAN_COLS - 1) / ST_MEAN_COLS, nmat), ST_MEAN_COLS, 0, st>>>(X, rowoff, idx, boff, K, p,
                                                                                              mean, zero_col);
    GG_CHECK_LAUNCH();
    const int nt = (p + ST_TT - 1) / ST_TT;
    dim3 grid(nt, nt, nmat);
    gg_count_launch(1);
    if ((p & 1) == 0) st_cov_kernel<true><<<grid, ST_THREADS, 0, st>>>(X, rowoff, idx, boff, K, p, mean, S);
    else st_cov_kernel<false><<<grid, ST_THREADS, 0, st>>>(X, rowoff, idx, boff, K, p, mean, S);
    GG_CHECK_LAUNCH();
    if (scale) {
        // the means are no longer needed: their workspace holds sqrt(diag)
        gg_count_launch(2);
        st_diag_kernel<<<st_blocks((size_t)nmat * p, 1), ST_THREADS, 0, st>>>(S, nmat, p, mean);
        GG_CHECK_LAUNCH();
        st_scale_kernel<<<dim3(st_blocks((size_t)p * p, nmat), nmat), ST_THREADS, 0, st>>>(S, p, mean);
        GG_CHECK_LAUNCH();
    }
    return 0;
}

int gg_launch_edge_count(const double* Theta, int nsub, int L, int K, int p, int* counts, cudaStream_t st)
{
    gg_count_launch(1);
    st_edge_count_kernel<<<dim3(st_blocks((size_t)p * p, L * K), L * K), ST_THREADS, 0, st>>>(Theta, nsub, L, K, p,
                                                                                                counts);
    GG_CHECK_LAUNCH();
    return 0;
}

int gg_launch_stars_instability(const int* counts, int L, int K, int p, int B, double* out, cudaStream_t st)
{
    gg_count_launch(1);
    st_instability_kernel<<<L * K, ST_THREADS, 0, st>>>(counts, p, B, out);
    GG_CHECK_LAUNCH();
    return 0;
}
