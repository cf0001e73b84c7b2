// gg_screen.cu -- exact component screen of the multiple graphical lasso (block_MGL).
//
// Entry (i, j), i != j, is an edge iff prox_P(s_ij) != 0, where s_ij = (n_k S_k,ij)_k and P is the per-entry penalty
// of the ADMM prox (GGL: l1 |.|_1 + l2 |.|_2; FGL: l1 |.|_1 + l2 chain TV).  prox_P(s) = 0 iff s lies in the
// subdifferential of P at 0, which is what the off-block KKT conditions of a block-diagonal solution need (Danaher,
// Wang & Witten 2014, section 5); so the MGL solution is block diagonal over the connected components of this graph.
//
// The prox is evaluated with prox_mgl_kernel's device routines and expressions at rho = 1 (compiled with -fmad=false),
// so the graph is the oracle's prox_p(n S) != 0 bit for bit, ties included.
//
// Output: upper-triangle bitmask, p rows of nw = ceil(p/32) words; bit b of word w in row i is column 32 w + b.  One
// warp per word, one thread per entry; the word is formed with a ballot (deterministic, no atomics).  The diagonal,
// the lower triangle and the tail bits past p are 0; lanes outside the strict upper triangle read nothing.
#include "gg_common.cuh"
#include "gg_condat.cuh"

#define SC_THREADS 256

template <int REG>
__global__ void __launch_bounds__(SC_THREADS)
mgl_screen_kernel(const double* __restrict__ S, const double* __restrict__ nk, double lambda1, double lambda2, int K,
                  int p, int nw, uint32_t* __restrict__ adj)
{
    extern __shared__ double ysm[];                  // FGL: K * SC_THREADS, [k][thread] (conflict free for the TV scan)
    const int lane = threadIdx.x & 31;
    const size_t word = (size_t)blockIdx.x * (SC_THREADS / 32) + (threadIdx.x >> 5);
    if (word >= (size_t)p * nw) return;              // whole warps only: the ballot below sees full warps
    const int i = (int)(word / nw), j = (int)(word - (size_t)i * nw) * 32 + lane;
    bool edge = false;
    if (j > i && j < p) {
        const size_t pp = (size_t)p * p, e = (size_t)i * p + j;
        if (REG == 0) {                              // group soft threshold of the l1-soft-thresholded vector
            double ss = 0.0;
            for (int k = 0; k < K; ++k) {
                const double s = nk ? nk[k] * S[k * pp + e] : S[k * pp + e];
                const double u = gg_soft(s, lambda1);
                ss += u * u;
            }
            const double nrm = sqrt(ss);
            const double a = nrm > lambda2 ? nrm : lambda2;
            const double f = a - lambda2;
            for (int k = 0; k < K; ++k) {
                const double s = nk ? nk[k] * S[k * pp + e] : S[k * pp + e];
                edge |= ((gg_soft(s, lambda1) * f) / a) != 0.0;
            }
        } else {                                     // TV prox across k, then l1 soft threshold
            double* y = ysm + threadIdx.x;
            for (int k = 0; k < K; ++k) y[k * SC_THREADS] = nk ? nk[k] * S[k * pp + e] : S[k * pp + e];
            gg_tv1d_inplace(y, K, SC_THREADS, lambda2);
            for (int k = 0; k < K; ++k) edge |= gg_soft(y[k * SC_THREADS], lambda1) != 0.0;
        }
    }
    const unsigned b = __ballot_sync(0xffffffffu, edge);
    if (lane == 0) adj[word] = b;
}

int gg_launch_mgl_screen(const double* S, const double* nk, double l1, double l2, int reg, int K, int p,
                         uint32_t* adj, cudaStream_t st)
{
    const int nw = (p + 31) / 32;
    const size_t words = (size_t)p * nw;
    const size_t blocks = (words + SC_THREADS / 32 - 1) / (SC_THREADS / 32);
    if (blocks > 0x7fffffffu) return -1;
    if (reg == 0) {
        gg_count_launch(1);
        mgl_screen_kernel<0><<<(unsigned)blocks, SC_THREADS, 0, st>>>(S, nk, l1, l2, K, p, nw, adj);
    } else {
        const size_t smem = (size_t)K * SC_THREADS * sizeof(double);
        if (smem > 200 * 1024) return -2;            // K too large for the shared-memory layout
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(mgl_screen_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)smem);
            if (e != cudaSuccess) return (int)e;
        }
        gg_count_launch(1);
        mgl_screen_kernel<1><<<(unsigned)blocks, SC_THREADS, smem, st>>>(S, nk, l1, l2, K, p, nw, adj);
    }
    GG_CHECK_LAUNCH();
    return 0;
}
