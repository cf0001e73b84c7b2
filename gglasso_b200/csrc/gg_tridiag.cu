// gg_tridiag.cu -- large-p symmetric eigensolver: Householder tridiagonalisation, tridiagonal
// divide & conquer, blocked back-transformation (sm_100a).  Batched over M matrices.
//
// Replaces np.linalg.eigh (LAPACK dsyevd) at admm_solver.py:181,199 / single_admm_solver.py:164,174
// for p > GG_SMALL_MAX.  Same three stages as dsyevd (dsytrd, dstedc, dormtr), laid out for the GPU:
//
//   1. sytrd   A = Q_H T Q_H^T.  Per column j two launches over the whole batch:
//              tr_col_kernel (one CTA per matrix: finish w_{j-1}, apply the pending rank-2 updates to row j
//              and form the Householder vector v_j) and tr_symv_kernel (streams the upper triangle of the
//              trailing matrix once: applies the pending rank-2 updates in registers, accumulates the full
//              y_j = A v_j from that half pass and stores the block only every q-th pass, see TR_QMAX).
//              The last TR_TAIL columns run in shared memory in one launch (tr_tail_kernel).
//   2. stedc   Cuppen divide & conquer with Gu/Eisenstat's stable eigenvector formula: rank-one tearing
//              at every split, leaves (<=32) by the shared-memory Jacobi kernel, then level-synchronous
//              merges: deflation (dc_prepare), secular equation (dc_secular, one warp per root),
//              Loewner z-hat (dc_zhat), eigenvectors of the rank-one update (dc_vectors) and the basis
//              update Qt_new = U^T Qt on FP64 tensor cores (dc_gemm, DMMA).
//   3. ormtr   Vt <- Vt Q_H^T with compact-WY panels (bt_larft_kernel, bt_apply_kernel, DMMA); every CTA owns a
//              band of rows and walks all panels, so the whole back-transformation is one launch.
//
// Eigenvectors are returned as rows (Vt), order arbitrary -- only V f(D) V^T is consumed downstream.
#include "gg_common.cuh"
#include "gg_jacobi_dev.cuh"
#include <stdlib.h>
#include <cmath>
#include <vector>

#define TR_EPS 2.220446049250313e-16
#define DC_LEAF 32
#define BT_NB 32
#define BT_R 32


// =============================================================================================
// stage 1: tridiagonalisation
// =============================================================================================
struct TrWs {
    double* Vh;      // (M,n,n) row j = Householder vector v_j (global indexing, v_j[j+1] = 1)
    double* tau;     // (M,n)
    double* d;       // (M,n)
    double* e;       // (M,n)
    double* vbuf;    // (M,2,n)
    double* w;       // (M,TR_QMAX,n) ring of the w vectors of the pending (not yet written back) rank-2 updates
    double* y;       // (M,n)
    int* cnt;        // (M) tile arrival counters of tr_step_kernel (zero between launches)
#ifdef TR_TIMING
    long long* dbg;  // (n,2,8) time stamps of one CTA per launch (instrumented build only; nullptr: no stamps)
#endif
};

#ifdef TR_TIMING
__device__ __forceinline__ long long tr_now()
{
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TR_STAMP(kind, slot) do { if (tr_stamp_on && ws.dbg) ws.dbg[((size_t)j * 2 + (kind)) * 8 + (slot)] = tr_now(); } while (0)
#else
#define TR_STAMP(kind, slot) do { } while (0)
#endif

// Lazy write-back of the rank-2 updates: the trailing block in memory may lag behind by up to TR_QMAX Householder
// steps.  Pass j re-applies the pending pairs (v_k, w_k), k in [kb, j-1], to each tile in registers (the same
// sequence of roundings as writing every pass), and only every q-th pass stores the tiles.  A read-only pass moves
// 8 B per element instead of 16.
#define TR_QMAX 4

__device__ __forceinline__ double tr_warp_allsum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum, result in every thread (fixed order => deterministic); one barrier; scratch >= 32 doubles
__device__ __forceinline__ double tr_block_allsum(double v, double* scratch)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = tr_warp_allsum(v);
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    return tr_warp_allsum(lane < nw ? scratch[lane] : 0.0);
}

// One CTA per matrix, step j in [0, n-1];  kb = first pending pair (pairs kb..j-1 are not yet applied to A in memory).
// Finishes w_{j-1} from the accumulated y, applies the pending updates to row j and forms the Householder vector
// v_j.  The step sits on the critical path of the launch chain, so every independent global load (row j, y,
// v_{j-1}) is issued up front into registers: the dependent chain is one memory round trip, two block reductions
// (one barrier each) and the stores.   Element i = j + tid + e*blockDim.x, e < EPT.
// (The body is shared by tr_col_kernel and by tr_step_kernel, where the CTA that finishes the last tile of a matrix
//  runs it for the next column: row j and y are then data written by other CTAs of the SAME grid, hence the
//  ld.global.cg loads -- L2 is the point of coherence, the fences are in tr_step_kernel.)
#ifdef TR_COL_PLAIN
#define TR_CLD(p) (*(p))
#else
#define TR_CLD(p) __ldcg(p)
#endif
template <int EPT, bool PREF>
__device__ __forceinline__ void tr_col_body(const double* A, int n, int j, int kb, const TrWs& ws, int m, int sk,
                                            bool stamp_on)
{
    __shared__ double red1[32], red2[32];
    __shared__ double s_a1;
#ifdef TR_TIMING
    const bool tr_stamp_on = stamp_on;
#endif
    const int tid = threadIdx.x, nt = blockDim.x;
    const double* rowj = A + (size_t)m * n * n + (size_t)j * n;
    const double* vprev = ws.vbuf + ((size_t)m * 2 + ((j + 1) & 1)) * n;    // v^{(j-1)}
    double* vcur = ws.vbuf + ((size_t)m * 2 + (j & 1)) * n;                 // v^{(j)}
    double* wring = ws.w + (size_t)m * TR_QMAX * n;
    const double* Vhm = ws.Vh + (size_t)m * n * n;
    double* y = ws.y + (size_t)m * n;
    double* tau = ws.tau + (size_t)m * n;
    const int cnt = j - kb;

    double a[EPT], yv[EPT], vp[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const int i = j + tid + e * nt;
        const bool ok = i < n;
        a[e] = ok ? TR_CLD(rowj + i) : 0.0;
        yv[e] = (ok && j >= 1) ? TR_CLD(y + i) : 0.0;
        vp[e] = (ok && j >= 1) ? vprev[i] : 0.0;
    }
    double tp = 0.0, yj = 0.0;
    if (j >= 1) { tp = tau[j - 1]; yj = TR_CLD(y + j); }
    // older pending pairs kb..j-2 (independent of w_{j-1}): a_i -= v_k[i] w_k[j] + w_k[i] v_k[j]
    // (PREF: fully unrolled with predicates so that all of these loads are in flight together with the ones above;
    //  the large-p variant keeps them in a loop -- no register spills in any kernel of the launch chain)
    if (!PREF) {
        if (sk) return;
        for (int q = 0; q < cnt - 1; ++q) {
            const int k = kb + q;
            const double* wk = wring + (size_t)(k % TR_QMAX) * n;
            const double* vk = Vhm + (size_t)k * n;
            const double wkj1 = wk[j], vkj1 = vk[j];
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int i = j + tid + e * nt;
                if (i < n) a[e] = a[e] - vk[i] * wkj1 - wk[i] * vkj1;
            }
        }
    } else {
        double wkj[TR_QMAX - 1], vkj[TR_QMAX - 1], wki[TR_QMAX - 1][EPT], vki[TR_QMAX - 1][EPT];
#pragma unroll
        for (int q = 0; q < TR_QMAX - 1; ++q) {
            const bool on = q < cnt - 1;
            const int k = on ? kb + q : 0;
            const double* wk = wring + (size_t)(k % TR_QMAX) * n;
            const double* vk = Vhm + (size_t)k * n;
            wkj[q] = on ? wk[j] : 0.0;
            vkj[q] = on ? vk[j] : 0.0;
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const int i = j + tid + e * nt;
                wki[q][e] = (on && i < n) ? wk[i] : 0.0;
                vki[q][e] = (on && i < n) ? vk[i] : 0.0;
            }
        }
        if (sk) return;                       // (block-uniform; no barrier has been passed yet)
        TR_STAMP(0, 2);
#pragma unroll
        for (int q = 0; q < TR_QMAX - 1; ++q)
#pragma unroll
            for (int e = 0; e < EPT; ++e)
                if (q < cnt - 1) a[e] = a[e] - vki[q][e] * wkj[q] - wki[q][e] * vkj[q];
    }
    if (j >= 1) {
        // w^{(j-1)} = p + alpha v, p = tau*y, alpha = -tau/2 * (p.v), on indices j..n-1;  v^{(j-1)}[j] = 1
        double part = 0.0;
#pragma unroll
        for (int e = 0; e < EPT; ++e) part += (tp * yv[e]) * vp[e];
        const double alpha = -0.5 * tp * tr_block_allsum(part, red1);      // (barrier: every read of y is done)
        TR_STAMP(0, 3);
        const double wj = tp * yj + alpha;
        double* w = wring + (size_t)((j - 1) % TR_QMAX) * n;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int i = j + tid + e * nt;
            if (i < n) {
                const double wi = tp * yv[e] + alpha * vp[e];
                w[i] = wi;
                a[e] = a[e] - vp[e] * wj - wi;
            }
        }
    }
    double part2 = 0.0;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const int i = j + tid + e * nt;
        if (i < n) y[i] = 0.0;        // consumed: clear for the atomics of the next tr_symv_kernel (indices > j)
        if (i < n && i >= j + 2) part2 += a[e] * a[e];
        if (i == j + 1 && i < n) s_a1 = a[e];
        if (i == j) ws.d[(size_t)m * n + j] = a[e];
    }
    const double xn2 = tr_block_allsum(part2, red2);
    TR_STAMP(0, 4);
    if (j < n - 1) {
        const double alpha = s_a1;
        double t = 0.0, beta = alpha, scale = 0.0;
        if (xn2 > 0.0) {
            beta = -copysign(sqrt(alpha * alpha + xn2), alpha);
            t = (beta - alpha) / beta;
            scale = 1.0 / (alpha - beta);
        }
        if (tid == 0) {
            tau[j] = t;
            ws.e[(size_t)m * n + j] = beta;
        }
        double* vh = ws.Vh + (size_t)m * n * n + (size_t)j * n;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int i = j + tid + e * nt;
            if (i < n && i >= j + 1) {
                const double v = (i == j + 1) ? 1.0 : a[e] * scale;
                vcur[i] = v;
                vh[i] = v;
            }
        }
    }
    TR_STAMP(0, 5);
}

template <int EPT, int THR, bool PREF>
__global__ void __launch_bounds__(THR)
tr_col_kernel(const double* A, int n, int j, int kb, TrWs ws, const int* __restrict__ skip)
{
    const int m = blockIdx.x;
#ifdef TR_TIMING
    const bool tr_stamp_on = (blockIdx.x == 0 && threadIdx.x == 0);
#endif
    TR_STAMP(0, 0);
    // Wait for the previous tr_symv_kernel first and only then release the next one: its CTAs start loading their
    // tiles of A before their own wait, which is safe exactly because the last writer of A has completed here.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
    TR_STAMP(0, 1);
    const int sk = skip ? skip[m] : 0;        // consumed in the body, after the other loads have been issued
    tr_col_body<EPT, PREF>(A, n, j, kb, ws, m, sk, blockIdx.x == 0 && threadIdx.x == 0);
}

// Streams the UPPER triangle of the trailing block, one CTA per 64x64 tile (I <= J): applies the pending rank-2
// updates kb..j-1 (a_rc -= v_k[r] w_k[c] + w_k[r] v_k[c]) in registers, stores the tile only on a write pass, and
// accumulates the full symmetric y = A v from that single pass: y_I += T v_J (row sums) and, mirrored,
// y_J += T^T v_I (column sums; strictly upper part on diagonal tiles).  Each thread owns a 4 x 4 register block
// (rows 4*ty+i, columns tx+16*jj: a half warp reads 128 contiguous bytes of a row); every global load of the CTA is
// issued before anything is consumed; partial sums go through shared memory, so the 128 FP64 atomics of a tile
// are four coalesced warp instructions.
// The kernel is instruction-issue bound (ncu: 55-66 % issue slots busy, FP64 pipe 15 %, DRAM 30 %), so the body is
// compiled twice: INTERIOR tiles (strictly above the diagonal and fully inside the block -- most of them) carry no
// bounds predicates, no masks and no selects.
#define SV_T 64
struct SvSmem {
    __align__(16) double vp[TR_QMAX][2][SV_T];
    __align__(16) double w[TR_QMAX][2][SV_T];
    __align__(16) double vI[SV_T];
    __align__(16) double vJ[SV_T];
    double rowp[SV_T][17];                       // [row][tx] partial row sums (stride 17: conflict-free read-back)
    double colp[16][SV_T];                       // [ty][col] partial column sums
};

// (Round 2 tried L2 cache-policy hints on these loads / stores -- evict_last for a pinned bottom-right part of every
//  matrix, evict_first for the rest: no gain for the chain, and the extra predicates in the unrolled load / store
//  loops cost 0.34 ms per tridiagonalisation at K=20, p=1000 even when switched off; removed.  The blocked path's
//  panel kernel keeps its own hints, where they are worth 3.5 ms.)
template <bool INTERIOR>
__device__ __forceinline__ void sv_tile_body(double* __restrict__ A, int n, int j, int kb, int write, const TrWs& ws,
                                             const int* __restrict__ skip, int m, int I, int J, SvSmem& sm,
                                             int pdl, bool& skipped)
{
    skipped = true;
    const int t = n - j - 1, base = j + 1, cnt = j - kb;
#ifdef TR_TIMING
    const bool tr_stamp_on = (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0);
#endif
    const int r0 = I * SV_T, c0 = J * SV_T;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int rb = r0 + 4 * ty, cb = c0 + tx;
    double* Am = A + (size_t)m * n * n + (size_t)base * n + base;
    double* pt = Am + (size_t)rb * n + cb;        // element (i, jj) of the register block: pt[i*n + 16*jj]
    // The tile is loaded BEFORE griddepcontrol.wait: A is written only by tr_symv_kernel launches, and the previous
    // one had completed before the column kernel in between released this grid (see tr_col_kernel), so these loads
    // overlap the column step.  ld.global.cg: straight from L2 -- no reuse, and no stale L1 lines across launches.
    // pdl 0 (tr_symv_kernel): as described above.  tr_step_kernel has no column kernel in between, so its grids wait
    // for their predecessor and only then release their successor (whose CTAs therefore never run beside a grid
    // older than their predecessor); pdl 1: the predecessor did not store A -- load early; pdl 2: it did -- wait first.
    if (pdl == 2) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;");
    }
    double a[4][4];
    unsigned okm = 0xffffu;
    if (INTERIOR) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) a[i][jj] = __ldcg(pt + (size_t)i * n + 16 * jj);
    } else {
        okm = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int r = rb + i, c = cb + 16 * jj;
                const bool ok = (r < t && c < t && c >= r);
                okm |= ok ? (1u << (4 * i + jj)) : 0u;
                a[i][jj] = ok ? __ldcg(pt + (size_t)i * n + 16 * jj) : 0.0;
            }
    }
    if (pdl != 2) asm volatile("griddepcontrol.wait;" ::: "memory");   // everything below reads what the column step wrote
    if (pdl == 1) asm volatile("griddepcontrol.launch_dependents;");
    TR_STAMP(1, 1);
    const int sk = skip ? skip[m] : 0;
    const double* vcur = ws.vbuf + ((size_t)m * 2 + (j & 1)) * n + base;
    const double* wring = ws.w + (size_t)m * TR_QMAX * n + base;
    const double* Vhm = ws.Vh + (size_t)m * n * n + base;
    double pv[2], pw[2], cv = 0.0;            // staged element e = tid + 256 u: pair q = e/128, half h, lane l
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int e = tid + 256 * u;
        const int q = e >> 7, h = (e >> 6) & 1, l = e & 63, k = kb + q;
        const int pos = (h ? c0 : r0) + l;
        const bool ok = (q < cnt) && (INTERIOR || pos < t);
        pv[u] = ok ? Vhm[(size_t)k * n + pos] : 0.0;
        pw[u] = ok ? wring[(size_t)(k % TR_QMAX) * n + pos] : 0.0;
    }
    if (tid < 2 * SV_T) {
        const int pos = (tid < SV_T) ? r0 + tid : c0 + tid - SV_T;
        cv = (INTERIOR || pos < t) ? vcur[pos] : 0.0;
    }
    if (sk) return;                           // (block-uniform; no barrier has been passed yet)
    skipped = false;
    TR_STAMP(1, 2);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int e = tid + 256 * u;
        (&sm.vp[0][0][0])[e] = pv[u];
        (&sm.w[0][0][0])[e] = pw[u];
    }
    if (tid < SV_T) sm.vI[tid] = cv;
    else if (tid < 2 * SV_T) sm.vJ[tid - SV_T] = cv;
    __syncthreads();
    TR_STAMP(1, 3);
    // pending updates, oldest first.  Out-of-range rows / columns carry zeros in the staged vectors, so only the
    // lower part of a diagonal tile has to be masked afterwards (it must stay zero for the sums below).
    for (int k = 0; k < cnt; ++k) {
        double wc[4], vc[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) { wc[jj] = sm.w[k][1][tx + 16 * jj]; vc[jj] = sm.vp[k][1][tx + 16 * jj]; }
        const double2 v01 = *reinterpret_cast<const double2*>(&sm.vp[k][0][4 * ty]);
        const double2 v23 = *reinterpret_cast<const double2*>(&sm.vp[k][0][4 * ty + 2]);
        const double2 w01 = *reinterpret_cast<const double2*>(&sm.w[k][0][4 * ty]);
        const double2 w23 = *reinterpret_cast<const double2*>(&sm.w[k][0][4 * ty + 2]);
        const double vr[4] = {v01.x, v01.y, v23.x, v23.y}, wr[4] = {w01.x, w01.y, w23.x, w23.y};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) a[i][jj] = a[i][jj] - vr[i] * wc[jj] - wr[i] * vc[jj];
    }
    if (!INTERIOR) {
        if (I == J && cnt > 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jj = 0; jj < 4; ++jj)
                    if (!(okm & (1u << (4 * i + jj)))) a[i][jj] = 0.0;
        }
    }
    if (write) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
                if (INTERIOR || (okm & (1u << (4 * i + jj)))) pt[(size_t)i * n + 16 * jj] = a[i][jj];
    }
#ifdef TR_TIMING
    if (a[0][0] == 1.2345e300) return;       // (forces the tile loads to have landed before the stamp)
#endif
    TR_STAMP(1, 4);
    {
        double vJ[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) vJ[q] = sm.vJ[tx + 16 * q];
        const double2 i01 = *reinterpret_cast<const double2*>(&sm.vI[4 * ty]);
        const double2 i23 = *reinterpret_cast<const double2*>(&sm.vI[4 * ty + 2]);
        const double vI[4] = {i01.x, i01.y, i23.x, i23.y};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double sacc = 0.0;
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) sacc = fma(a[i][jj], vJ[jj], sacc);
            sm.rowp[4 * ty + i][tx] = sacc;              // includes the diagonal
        }
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            double sacc = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const bool dg = !INTERIOR && (I == J) && (rb + i == cb + 16 * jj);   // mirrored part: strictly upper
                sacc = fma(dg ? 0.0 : a[i][jj], vI[i], sacc);
            }
            sm.colp[ty][tx + 16 * jj] = sacc;
        }
    }
    __syncthreads();
    TR_STAMP(1, 5);
    double* y = ws.y + (size_t)m * n + base;
    if (tid < SV_T) {
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int q = 0; q < 16; q += 2) { s0 += sm.rowp[tid][q]; s1 += sm.rowp[tid][q + 1]; }
        if (INTERIOR || r0 + tid < t) atomicAdd(y + r0 + tid, s0 + s1);
    } else if (tid < 2 * SV_T) {
        const int cc = tid - SV_T;
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int q = 0; q < 16; q += 2) { s0 += sm.colp[q][cc]; s1 += sm.colp[q + 1][cc]; }
        if (INTERIOR || c0 + cc < t) atomicAdd(y + c0 + cc, s0 + s1);
    }
    TR_STAMP(1, 6);
}

// (256, 3): 80 registers, no spills.  (256, 4) -- 64 registers, 28 bytes of spills -- was 3 % faster on a single
// stream but produced non-finite eigenvalues for single matrices when five host threads drove five solves
// concurrently (bisected on the B200, DESIGN.md 4.4); not understood, so not used.
#ifndef SV_MINB
#define SV_MINB 3
#endif
__global__ void __launch_bounds__(256, SV_MINB)
tr_symv_kernel(double* __restrict__ A, int n, int j, int kb, int write, TrWs ws, const int* __restrict__ skip, int nt)
{
    __shared__ SvSmem sm;
    // Boustrophedon sweep: consecutive launches walk the (matrix, tile) space in opposite directions, so a launch
    // starts with the tiles the previous one touched last -- they are still in L2 (an identical sweep order is the
    // worst case for an LRU-like cache when the ~80 MB working set exceeds the usable capacity).
    const bool rev = (j & 1) != 0;
    const int m = rev ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y;
    int idx = rev ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x, I = 0;
    while (idx >= nt - I) { idx -= nt - I; ++I; }
    const int J = I + idx;
#ifdef TR_TIMING
    const bool tr_stamp_on = (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0);
#endif
    TR_STAMP(1, 0);
    asm volatile("griddepcontrol.launch_dependents;");       // let the next grid in the chain become resident
    const bool interior = (I < J) && ((J + 1) * SV_T <= n - j - 1);
    bool skipped;
    if (interior) sv_tile_body<true>(A, n, j, kb, write, ws, skip, m, I, J, sm, 0, skipped);
    else sv_tile_body<false>(A, n, j, kb, write, ws, skip, m, I, J, sm, 0, skipped);
}

// tr_symv_kernel(j) followed, in the same launch, by the column step j+1 (tr_col_body): the CTA that finishes the last
// tile of a matrix -- found with a per-matrix arrival counter -- runs it, so a column costs ONE launch boundary instead
// of two and the column steps of all matrices but the last to finish are hidden behind the tile work of the others.
// Ordering: every thread fences its atomics on y / stores of A before the CTA's arrival; the last CTA fences again
// before it reads y and row j+1 (ld.global.cg).  col_next = 0 on the last chain step (tr_tail_kernel continues).
__global__ void __launch_bounds__(256, 3)
tr_step_kernel(double* A, int n, int j, int kb, int write, TrWs ws, const int* __restrict__ skip, int nt,
               int early, int col_next)
{
    __shared__ SvSmem sm;
    __shared__ int s_last;
    const bool rev = (j & 1) != 0;
    const int m = rev ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y;
    int idx = rev ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x, I = 0;
    while (idx >= nt - I) { idx -= nt - I; ++I; }
    const int J = I + idx;
#ifdef TR_TIMING
    const bool tr_stamp_on = (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0);
#endif
    TR_STAMP(1, 0);
    const bool interior = (I < J) && ((J + 1) * SV_T <= n - j - 1);
    bool skipped;
    if (interior) sv_tile_body<true>(A, n, j, kb, write, ws, skip, m, I, J, sm, early ? 1 : 2, skipped);
    else sv_tile_body<false>(A, n, j, kb, write, ws, skip, m, I, J, sm, early ? 1 : 2, skipped);
    if (skipped || !col_next) return;         // (block-uniform)
    __syncthreads();
    if (threadIdx.x == 0) {
        // release (cumulative over the CTA's atomics and stores, ordered by the barrier) / acquire in one RMW
        int prev;
        asm volatile("atom.add.acq_rel.gpu.global.s32 %0, [%1], 1;" : "=r"(prev) : "l"(ws.cnt + m) : "memory");
        s_last = (prev == (int)gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    if (threadIdx.x == 0) ws.cnt[m] = 0;
    const int jn = j + 1, kbn = write ? j : kb, len = n - jn;
    if (len <= 512) tr_col_body<2, true>(A, n, jn, kbn, ws, m, 0, false);
    else if (len <= 1024) tr_col_body<4, false>(A, n, jn, kbn, ws, m, 0, false);
    else tr_col_body<8, false>(A, n, jn, kbn, ws, m, 0, false);
}

// Tail of the tridiagonalisation: once the trailing block has at most TR_TAIL rows it fits in shared memory, and
// one CTA per matrix finishes all remaining columns in a single launch (block barriers instead of ~2*TR_TAIL
// dependent kernel launches).  Takes over at column js: finishes w_{js-1} from the accumulated y, loads the
// upper triangle of the trailing block with the pending rank-2 update applied (mirrored into a full symmetric
// tile), then runs the unblocked Householder steps in place.
#define TR_TAIL 144
__global__ void __launch_bounds__(512)
tr_tail_kernel(const double* __restrict__ A, int n, int js, TrWs ws, const int* __restrict__ skip, int pending)
{
    extern __shared__ double tsm[];
    const int m = blockIdx.x;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (skip && skip[m]) return;
    const int ts = n - js, ld = ts | 1;
    double* B = tsm;                      // ts x ld
    double* vv = tsm + (size_t)ts * ld;   // ts
    double* ww = vv + ts;                 // ts
    double* yy = ww + ts;                 // ts
    double* red = yy + ts;                // 64
    double* bc = red + 64;                // 4
    const int tid = threadIdx.x, nt = blockDim.x;
    const double* Am = A + (size_t)m * n * n;
    double* tau = ws.tau + (size_t)m * n;
    double* dd = ws.d + (size_t)m * n;
    double* ee = ws.e + (size_t)m * n;
    double* Vh = ws.Vh + (size_t)m * n * n;
    const bool pend = js >= 1 && pending;      // blocked path: the trailing block is fully updated, nothing pending
    if (pend) {
        const double* y = ws.y + (size_t)m * n;
        const double* vprev = ws.vbuf + ((size_t)m * 2 + ((js + 1) & 1)) * n;
        const double tp = tau[js - 1];
        double part[1] = {0.0};
        for (int r = tid; r < ts; r += nt) part[0] += (tp * y[js + r]) * vprev[js + r];
        gg_block_sum<1>(part, red);
        if (tid == 0) bc[0] = -0.5 * tp * part[0];
        __syncthreads();
        const double alpha = bc[0];
        for (int r = tid; r < ts; r += nt) {
            vv[r] = vprev[js + r];
            ww[r] = tp * y[js + r] + alpha * vprev[js + r];
        }
        __syncthreads();
    }
    for (int idx = tid; idx < ts * ts; idx += nt) {
        const int r = idx / ts, c = idx - r * ts;
        const int rr = r < c ? r : c, cc = r < c ? c : r;
        double a = Am[(size_t)(js + rr) * n + js + cc];
        if (pend) a = a - vv[rr] * ww[cc] - ww[rr] * vv[cc];
        B[r * ld + c] = a;
    }
    __syncthreads();
    for (int jj = 0; jj < ts; ++jj) {
        const int j = js + jj, len = ts - jj - 1;
        if (tid == 0) dd[j] = B[jj * ld + jj];
        if (len == 0) break;
        const double* x = B + (size_t)jj * ld + jj + 1;          // row jj to the right of the diagonal
        double part[1] = {0.0};
        for (int i = 1 + tid; i < len; i += nt) part[0] += x[i] * x[i];
        gg_block_sum<1>(part, red);
        if (tid == 0) {
            const double alpha = x[0], xn2 = part[0];
            double t = 0.0, beta = alpha, scale = 0.0;
            if (xn2 > 0.0) {
                beta = -copysign(sqrt(alpha * alpha + xn2), alpha);
                t = (beta - alpha) / beta;
                scale = 1.0 / (alpha - beta);
            }
            tau[j] = t; ee[j] = beta; bc[1] = scale; bc[2] = t;
        }
        __syncthreads();
        const double scale = bc[1], tj = bc[2];
        for (int i = tid; i < len; i += nt) {
            const double v = (i == 0) ? 1.0 : x[i] * scale;
            vv[i] = v;
            Vh[(size_t)j * n + j + 1 + i] = v;
        }
        __syncthreads();
        // y = B22 v  (two threads per row, even / odd columns)
        {
            const int r = tid >> 1, h = tid & 1;
            double s = 0.0;
            if (r < len) {
                const double* row = B + (size_t)(jj + 1 + r) * ld + jj + 1;
                for (int c = h; c < len; c += 2) s = fma(row[c], vv[c], s);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            if (r < len && h == 0) yy[r] = s;
        }
        __syncthreads();
        double dp[1] = {0.0};
        for (int i = tid; i < len; i += nt) dp[0] += (tj * yy[i]) * vv[i];
        gg_block_sum<1>(dp, red);
        if (tid == 0) bc[3] = -0.5 * tj * dp[0];
        __syncthreads();
        const double al = bc[3];
        for (int i = tid; i < len; i += nt) ww[i] = tj * yy[i] + al * vv[i];
        __syncthreads();
        {
            const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
            for (int r = wid; r < len; r += nw) {
                double* row = B + (size_t)(jj + 1 + r) * ld + jj + 1;
                const double vr = vv[r], wr = ww[r];
                for (int c = lane; c < len; c += 32) row[c] -= vr * ww[c] + wr * vv[c];
            }
        }
        __syncthreads();
    }
}

#include "gg_sytrd_blocked.cuh"

// =============================================================================================
// stage 2: divide & conquer on the tridiagonal matrices
// =============================================================================================
struct DcWs {
    double* lam[2];   // (M,n) eigenvalues, ping-pong
    double* z;        // (M,n)
    double* dl;       // (M,n) non-deflated poles (ascending) per node
    double* wnd;      // (M,n) their z components
    double* zhat;     // (M,n)
    int* ndrow;       // (M,n) global row of the i-th non-deflated vector
    double* rotc;     // (M,n) Givens rotations of the deflation step (cos, sin, row pair)
    double* rots;     // (M,n)
    int* rotp;        // (M,n)
    int* rotn;        // (M,n)
    int* nodek;       // (M,nodes_max) number of non-deflated
    int* nodeka;      // (M,nodes_max,2) lengths of the two per-child K lists below
    int* lista;       // (M,n) non-deflated poles whose row of Qt has entries in the first child's columns
    int* listb;       // (M,n) ... in the second child's columns (rows mixed by a Givens deflation are in both)
    int* dfl;         // (M,n) deflated rows of every node, in output order (read by dc_copy_deflated_kernel)
    int* nodendf;     // (M,nodes_max) their number
    double* noderho;  // (M,nodes_max)
    double* U;        // (M,n,n) Delta / eigenvector matrices, block diagonal like Qt
    int nodes_max;
};

// Reciprocal for the secular equation: hardware seed (about 20 bits) plus two Newton steps, no special-case
// handling -- about 6 instructions instead of the ~35 of an IEEE division, and dc_secular_kernel is bound by
// exactly that instruction count.  Accurate to an ulp or two, which the stopping test's rounding bound
// (8 sum|t| eps) covers; the pole distances that define the eigenvectors are formed without any division.
__device__ __forceinline__ double dc_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
}

__host__ __device__ __forceinline__ int dc_bnd(int n, int level, int i) { return (int)(((long long)i * n) >> level); }

// normalise T to unit max-norm (as dstedc does) so the deflation tolerance is scale free
__global__ void __launch_bounds__(256)
dc_scale_kernel(double* __restrict__ d, double* __restrict__ e, int n, double* __restrict__ scale,
                const int* __restrict__ skip)
{
    __shared__ double red[32];
    __shared__ double s_inv;
    const int m = blockIdx.x;
    if (skip && skip[m]) return;
    double mx = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) {
        mx = fmax(mx, fabs(d[(size_t)m * n + i]));
        if (i < n - 1) mx = fmax(mx, fabs(e[(size_t)m * n + i]));
    }
    mx = gg_block_max(mx, red);
    if (threadIdx.x == 0) {
        if (!(mx > 0.0)) mx = 1.0;
        scale[m] = mx;
        s_inv = 1.0 / mx;
    }
    __syncthreads();
    const double inv = s_inv;
    for (int i = threadIdx.x; i < n; i += 256) {
        d[(size_t)m * n + i] *= inv;
        if (i < n - 1) e[(size_t)m * n + i] *= inv;
    }
}

__global__ void dc_unscale_kernel(const double* __restrict__ lam, const double* __restrict__ scale, int n,
                                  double* __restrict__ D, const int* __restrict__ skip)
{
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    const double s = scale[m];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        D[(size_t)m * n + i] = lam[(size_t)m * n + i] * s;
}

// subtract |e_s| from both neighbours of every split point (all levels at once)
__global__ void dc_tear_kernel(double* __restrict__ d, const double* __restrict__ e, int n, int levels,
                               const int* __restrict__ skip)
{
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;   // enumerates (level, node)
    int l = 0, i = t;
    while (l < levels && i >= (1 << l)) { i -= (1 << l); ++l; }
    if (l >= levels) return;
    const int s = dc_bnd(n, l + 1, 2 * i + 1);
    const double rho = fabs(e[(size_t)m * n + s - 1]);
    d[(size_t)m * n + s - 1] -= rho;
    d[(size_t)m * n + s] -= rho;
}

// leaves: dense (<= DC_LEAF) tridiagonal blocks by shared-memory Jacobi; writes lam, block-diagonal Qt
__global__ void __launch_bounds__(128)
dc_leaf_kernel(const double* __restrict__ d, const double* __restrict__ e, int n, int levels,
               double* __restrict__ lam, double* __restrict__ Qt, const int* __restrict__ skip)
{
    __shared__ double G[DC_LEAF * (DC_LEAF + 1)];
    __shared__ double s_sigma;
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    const int lo = dc_bnd(n, levels, blockIdx.x), hi = dc_bnd(n, levels, blockIdx.x + 1);
    const int sz = hi - lo, ld = DC_LEAF + 1;
    const double* dm = d + (size_t)m * n;
    const double* em = e + (size_t)m * n;
    for (int idx = threadIdx.x; idx < sz * sz; idx += blockDim.x) {
        const int r = idx / sz, c = idx % sz;
        double v = 0.0;
        if (r == c) v = dm[lo + r];
        else if (c == r + 1) v = em[lo + r];
        else if (r == c + 1) v = em[lo + c];
        G[r * ld + c] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double lo_b = 1.0e300, hi_b = -1.0e300;
        for (int r = 0; r < sz; ++r) {
            double rs = 0.0;
            if (r > 0) rs += fabs(G[r * ld + r - 1]);
            if (r + 1 < sz) rs += fabs(G[r * ld + r + 1]);
            lo_b = fmin(lo_b, G[r * ld + r] - rs);
            hi_b = fmax(hi_b, G[r * ld + r] + rs);
        }
        const double c = 0.5 * (lo_b + hi_b);
        double h = 0.5 * (hi_b - lo_b);
        if (!(h > 0.0)) h = fmax(fabs(c), 1.0);
        s_sigma = 2.0 * h - c;
    }
    __syncthreads();
    const double sigma = s_sigma;
    if (threadIdx.x < sz) G[threadIdx.x * ld + threadIdx.x] += sigma;
    __syncthreads();
    jacobi_rows_smem<8, DC_LEAF / 8>(G, sz, ld, 4.0e-15, 40);
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int r = wid; r < sz; r += 4) {
        const double x = (lane < sz) ? G[r * ld + lane] : 0.0;
        const double nrm = sqrt(gg_warp_sum(x * x));
        if (lane == 0) lam[(size_t)m * n + lo + r] = nrm - sigma;
        if (lane < sz) Qt[(size_t)m * n * n + (size_t)(lo + r) * n + lo + lane] = x / nrm;
    }
}

// exclusive prefix sum of one int per thread over the block (<= 1024 threads); total in *tot.  scratch: 33 ints
__device__ __forceinline__ int dc_block_excl_scan(int v, int* scratch, int* tot)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) scratch[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int w = lane < nw ? scratch[lane] : 0;
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += u;
        }
        scratch[lane] = wi - w;                  // exclusive offset of warp `lane`
        if (lane == 31) scratch[32] = wi;
    }
    __syncthreads();
    const int res = scratch[wid] + incl - v;
    *tot = scratch[32];
    __syncthreads();                             // scratch may be reused by the caller
    return res;
}

// One CTA per node: z vector, sort, deflation, Givens rotations on rows, eigenvalues of the deflated pairs.
// Deflation runs in parallel under the assumption that no two poles are close enough to be rotated into each
// other (dlaed2's second criterion): small z components are flagged, the survivors compacted with block scans, every
// neighbouring pair of survivors is tested, and only if a pair fails the test thread 0 redoes the merge with the
// serial scan (identical results by construction: without a rotation the serial scan produces exactly these lists).
// The deflated rows are copied by dc_copy_deflated_kernel (many CTAs) instead of this one-CTA-per-node kernel.
__global__ void __launch_bounds__(1024)
dc_prepare_kernel(const double* __restrict__ e, int n, int level, const double* __restrict__ lam_in,
                  double* __restrict__ lam_out, double* __restrict__ Qin, double* __restrict__ Qout, DcWs ws,
                  const int* __restrict__ skip)
{
    extern __shared__ double sm[];             // d[N], z[N], then ints idx[N], nd[N], df[N]
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    const int node = blockIdx.x;
    const int lo = dc_bnd(n, level, node), hi = dc_bnd(n, level, node + 1), mid = dc_bnd(n, level + 1, 2 * node + 1);
    const int N = hi - lo, n1 = mid - lo;
    double* sd = sm;
    double* sz = sm + N;
    int* idx = (int*)(sm + 2 * N);
    int* nd = idx + N;
    int* df = nd + N;
    unsigned char* typ = (unsigned char*)(df + N);   // 1: first child, 3: second child, 2: mixed by a rotation
    double* rc = ws.rotc + (size_t)m * n + lo;  // rotation lists live in global memory (only thread 0 writes)
    double* rs = ws.rots + (size_t)m * n + lo;
    int* rp = ws.rotp + (size_t)m * n + lo;
    int* rn = ws.rotn + (size_t)m * n + lo;
    __shared__ int s_k, s_ndf, s_nrot;
    __shared__ double s_rho, s_red[64], s_max[2];
    const int tid = threadIdx.x, nt = blockDim.x;
    double* Qm = Qin + (size_t)m * n * n;
    const double es = e[(size_t)m * n + mid - 1];
    const double sgn = es >= 0.0 ? 1.0 : -1.0;
    const double rho = 2.0 * fabs(es);
    const double isq2 = 0.70710678118654752440;
    for (int i = tid; i < N; i += nt) {
        sd[i] = lam_in[(size_t)m * n + lo + i];
        sz[i] = (i < n1 ? Qm[(size_t)(lo + i) * n + mid - 1] : sgn * Qm[(size_t)(lo + i) * n + mid]) * isq2;
        typ[i] = (i < n1) ? 1 : 3;
    }
    __syncthreads();
    // rank sort (stable)
    for (int i = tid; i < N; i += nt) {
        const double di = sd[i];
        int r = 0;
        for (int q = 0; q < N; ++q) {
            const double dq = sd[q];
            r += (dq < di || (dq == di && q < i)) ? 1 : 0;
        }
        idx[r] = i;
    }
    __syncthreads();
    {
        double dm = 0.0, zm = 0.0;
        for (int i = tid; i < N; i += nt) { dm = fmax(dm, fabs(sd[i])); zm = fmax(zm, fabs(sz[i])); }
        dm = gg_block_max(dm, s_red);
        __syncthreads();
        zm = gg_block_max(zm, s_red + 32);
        if (tid == 0) { s_max[0] = dm; s_max[1] = zm; }
    }
    __syncthreads();
    __shared__ int s_scan[33];
    int* la = ws.lista + (size_t)m * n + lo;
    int* lb = ws.listb + (size_t)m * n + lo;
    bool serial = true;
    {
        const double dmax = s_max[0], zmax = s_max[1];
        const double tol = 8.0 * TR_EPS * fmax(dmax, zmax);
        if (!(rho * zmax <= tol)) {
            const int C = (N + nt - 1) / nt;
            const int t0 = min(N, tid * C), t1 = min(N, t0 + C);
            int cs = 0;
            for (int t = t0; t < t1; ++t) cs += (rho * fabs(sz[idx[t]]) <= tol) ? 1 : 0;
            int ndf_p;
            const int off = dc_block_excl_scan(cs, s_scan, &ndf_p);
            int sp = off, cp = t0 - off;
            for (int t = t0; t < t1; ++t) {
                const int nj = idx[t];
                if (rho * fabs(sz[nj]) <= tol) df[sp++] = nj;
                else nd[cp++] = nj;
            }
            __syncthreads();
            const int k_p = N - ndf_p;
            int trig = 0;
            for (int c = tid + 1; c < k_p; c += nt) {
                const int pj = nd[c - 1], nj = nd[c];
                const double sv = sz[pj], cv = sz[nj];
                const double den = cv * cv + sv * sv;
                const double tt = sd[nj] - sd[pj];
                trig |= (fabs(tt * cv * sv) <= tol * den) ? 1 : 0;
            }
            if (!__syncthreads_or(trig)) {
                serial = false;
                // K lists of the two children (no rotation: every pole belongs to exactly one child)
                const int C2 = (k_p + nt - 1) / nt;
                const int c0 = min(k_p, tid * C2), c1 = min(k_p, c0 + C2);
                int ca = 0;
                for (int c = c0; c < c1; ++c) ca += (typ[nd[c]] != 3) ? 1 : 0;
                int ka_p;
                const int offa = dc_block_excl_scan(ca, s_scan, &ka_p);
                int pa = offa, pb = c0 - offa;
                for (int c = c0; c < c1; ++c) {
                    if (typ[nd[c]] != 3) la[pa++] = c;
                    else lb[pb++] = c;
                }
                if (tid == 0) {
                    ws.nodeka[((size_t)m * ws.nodes_max + node) * 2] = ka_p;
                    ws.nodeka[((size_t)m * ws.nodes_max + node) * 2 + 1] = k_p - ka_p;
                    s_k = k_p; s_ndf = ndf_p; s_nrot = 0; s_rho = rho;
                    ws.nodek[(size_t)m * ws.nodes_max + node] = k_p;
                    ws.noderho[(size_t)m * ws.nodes_max + node] = rho;
                }
            }
        }
    }
    if (serial && tid == 0) {
        const double dmax = s_max[0], zmax = s_max[1];
        const double tol = 8.0 * TR_EPS * fmax(dmax, zmax);
        int k = 0, ndf = 0, nrot = 0, pj = -1;
        if (rho * zmax <= tol) {
            for (int i = 0; i < N; ++i) df[ndf++] = i;
        } else {
            for (int t = 0; t < N; ++t) {
                const int nj = idx[t];
                if (rho * fabs(sz[nj]) <= tol) { df[ndf++] = nj; continue; }
                if (pj < 0) { pj = nj; continue; }
                double s = sz[pj], c = sz[nj];
                const double den = c * c + s * s;                // |z| <= 1 after normalisation: no overflow
                const double tt = sd[nj] - sd[pj];
                // |t c s| <= tol with c = z_nj/tau, s = -z_pj/tau, tau^2 = den: tested without the square root and
                // the division, which are only needed for the (rare) rotation -- this loop is one serial thread
                if (fabs(tt * c * s) <= tol * den) {
                    const double tau = sqrt(den);
                    const double itau = 1.0 / tau;
                    c *= itau; s = -s * itau;
                    sz[nj] = tau; sz[pj] = 0.0;
                    rp[nrot] = pj; rn[nrot] = nj; rc[nrot] = c; rs[nrot] = s; ++nrot;
                    const double tnew = sd[pj] * c * c + sd[nj] * s * s;
                    sd[nj] = sd[pj] * s * s + sd[nj] * c * c;
                    sd[pj] = tnew;
                    df[ndf++] = pj;
                    if (typ[pj] != typ[nj]) typ[nj] = 2;
                    pj = nj;
                } else {
                    nd[k++] = pj;
                    pj = nj;
                }
            }
            if (pj >= 0) nd[k++] = pj;
        }
        // The rows of Qt are block diagonal (each child's eigenvectors live in its own columns), so the basis update
        // of a column range only needs the poles whose row has entries there: two K lists, as dlaed3's coltyp split
        int ka = 0, kb = 0;
        for (int i = 0; i < k; ++i) {
            const int ty = typ[nd[i]];
            if (ty != 3) la[ka++] = i;
            if (ty != 1) lb[kb++] = i;
        }
        ws.nodeka[((size_t)m * ws.nodes_max + node) * 2] = ka;
        ws.nodeka[((size_t)m * ws.nodes_max + node) * 2 + 1] = kb;
        s_k = k; s_ndf = ndf; s_nrot = nrot; s_rho = rho;
        ws.nodek[(size_t)m * ws.nodes_max + node] = k;
        ws.noderho[(size_t)m * ws.nodes_max + node] = rho;
    }
    __syncthreads();
    __threadfence_block();
    const int k = s_k, ndf = s_ndf, nrot = s_nrot;
    // Givens rotations on row pairs (in order; chains share rows)
    for (int r = 0; r < nrot; ++r) {
        double* a = Qm + (size_t)(lo + rp[r]) * n + lo;
        double* b = Qm + (size_t)(lo + rn[r]) * n + lo;
        const double c = rc[r], s = rs[r];
        for (int col = tid; col < N; col += nt) {
            const double x = a[col], yv = b[col];
            a[col] = c * x + s * yv;
            b[col] = -s * x + c * yv;
        }
        __syncthreads();
    }
    for (int i = tid; i < k; i += nt) {
        ws.ndrow[(size_t)m * n + lo + i] = lo + nd[i];
        ws.dl[(size_t)m * n + lo + i] = sd[nd[i]];
        ws.wnd[(size_t)m * n + lo + i] = sz[nd[i]];
    }
    // deflated eigenpairs go to rows lo+k.. of the output unchanged: eigenvalues here, rows in dc_copy_deflated_kernel
    int* dfl = ws.dfl + (size_t)m * n + lo;
    for (int t = tid; t < ndf; t += nt) {
        dfl[t] = df[t];
        lam_out[(size_t)m * n + lo + k + t] = sd[df[t]];
    }
    if (tid == 0) ws.nodendf[(size_t)m * ws.nodes_max + node] = ndf;
}

// Qout[lo+k+t][lo..hi) = Qin[lo+dfl[t]][lo..hi): one warp per deflated row.  grid (ceil(Nmax/8), nodes, M)
__global__ void __launch_bounds__(256)
dc_copy_deflated_kernel(int n, int level, const double* __restrict__ Qin, double* __restrict__ Qout, DcWs ws,
                        const int* __restrict__ skip)
{
    const int m = blockIdx.z;
    if (skip && skip[m]) return;
    const int node = blockIdx.y;
    const int ndf = ws.nodendf[(size_t)m * ws.nodes_max + node];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int t = blockIdx.x * 8 + wid;
    if (t >= ndf) return;
    const int k = ws.nodek[(size_t)m * ws.nodes_max + node];
    const int lo = dc_bnd(n, level, node), N = dc_bnd(n, level, node + 1) - lo;
    const double* src = Qin + (size_t)m * n * n + (size_t)(lo + ws.dfl[(size_t)m * n + lo + t]) * n + lo;
    double* dst = Qout + (size_t)m * n * n + (size_t)(lo + k + t) * n + lo;
    for (int col = lane; col < N; col += 128) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (col + 32 * u < N) ? src[col + 32 * u] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (col + 32 * u < N) dst[col + 32 * u] = v[u];
    }
}

// One warp per root: solves 1 + rho sum w_i^2/(dl_i - lam) = 0 in (dl_j, dl_{j+1}) with the shift to the
// nearer pole, rational ("middle way") steps safeguarded by bisection; writes Delta[j][i] = dl_i - lam_j.
__global__ void __launch_bounds__(256)
dc_secular_kernel(int n, int level, double* __restrict__ lam_out, DcWs ws, const int* __restrict__ skip)
{
    extern __shared__ double sm[];           // dl[k], w2[k]
    const int m = blockIdx.z;
    if (skip && skip[m]) return;
    const int node = blockIdx.y;
    const int k = ws.nodek[(size_t)m * ws.nodes_max + node];
    if ((int)blockIdx.x * 8 >= k) return;
    const int lo = dc_bnd(n, level, node);
    const double rho = ws.noderho[(size_t)m * ws.nodes_max + node];
    double* sdl = sm;
    double* sw2 = sm + k;
    for (int i = threadIdx.x; i < k; i += 256) {
        sdl[i] = ws.dl[(size_t)m * n + lo + i];
        const double w = ws.wnd[(size_t)m * n + lo + i];
        sw2[i] = rho * w * w;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int j = blockIdx.x * 8 + wid;
    if (j >= k) return;
    double* Drow = ws.U + (size_t)m * n * n + (size_t)(lo + j) * n + lo;
    int org;
    double tau;
    if (k == 1) {
        org = 0; tau = sw2[0];
    } else {
        const bool last = (j == k - 1);
        double lb, ub;
        int ia, ib;
        if (!last) {
            const double delta = sdl[j + 1] - sdl[j], mid = 0.5 * delta;
            double rest = 0.0;                       // all poles but the two that bracket the root, at the midpoint
            for (int i = lane; i < k; i += 32)
                if (i != j && i != j + 1) rest += sw2[i] * dc_rcp((sdl[i] - sdl[j]) - mid);
            const double c0 = 1.0 + gg_warp_sum(rest);
            const double wj = sw2[j], wj1 = sw2[j + 1];
            const double f = c0 + (wj1 - wj) / mid;
            // initial guess as in dlaed4: keep the two bracketing poles exact, freeze the rest at its midpoint value,
            // and take the root of the resulting quadratic on the side of the origin
            if (f >= 0.0) {
                org = j; lb = 0.0; ub = mid;
                const double a = c0 * delta + wj + wj1, b = wj * delta;
                const double sq = sqrt(fabs(a * a - 4.0 * b * c0));
                tau = (a > 0.0) ? 2.0 * b / (a + sq) : (a - sq) / (2.0 * c0);
            } else {
                org = j + 1; lb = -mid; ub = 0.0;
                const double a = -c0 * delta + wj + wj1, b = wj1 * delta;
                const double sq = sqrt(fabs(a * a + 4.0 * b * c0));
                tau = (a > 0.0) ? -2.0 * b / (a + sq) : (a - sq) / (2.0 * c0);   // the negative root of c0 t^2 - a t - b
            }
            if (!(tau > lb && tau < ub)) tau = 0.5 * (lb + ub);      // also catches NaN
            ia = j; ib = j + 1;
        } else {
            double span = 0.0;
            for (int i = lane; i < k; i += 32) span += sw2[i];
            span = gg_warp_sum(span);
            org = k - 1; lb = 0.0; ub = span; tau = 0.5 * span; ia = k - 2; ib = k - 1;
        }
        const double dorg = sdl[org];
        const int split = last ? (k - 1) : (j + 1);          // psi: i < split, phi: i >= split
        for (int it = 0; it < 100; ++it) {
            double psi = 0.0, phi = 0.0, dpsi = 0.0, dphi = 0.0, sabs = 0.0;
            for (int i = lane; i < k; i += 32) {
                const double rcp = dc_rcp((sdl[i] - dorg) - tau);      // one reciprocal per term
                const double t = sw2[i] * rcp;
                const double dt = t * rcp;
                if (i < split) { psi += t; dpsi += dt; } else { phi += t; dphi += dt; }
                sabs += fabs(t);
            }
            psi = gg_warp_sum(psi); phi = gg_warp_sum(phi); dpsi = gg_warp_sum(dpsi);
            dphi = gg_warp_sum(dphi); sabs = gg_warp_sum(sabs);
            const double f = 1.0 + psi + phi, df = dpsi + dphi;
            if (fabs(f) <= TR_EPS * (8.0 * sabs + 2.0 + fabs(tau) * df)) break;
            if (f < 0.0) lb = fmax(lb, tau); else ub = fmin(ub, tau);
            const double Da = (sdl[ia] - dorg) - tau, Db = (sdl[ib] - dorg) - tau;
            const double c = f - Da * dpsi - Db * dphi;
            const double a = (Da + Db) * f - Da * Db * df;
            const double b = Da * Db * f;
            double eta = 0.0;
            bool ok = false;
            if (c == 0.0) {
                if (a != 0.0) { eta = b / a; ok = true; }
            } else {
                const double disc = a * a - 4.0 * b * c;
                if (disc >= 0.0) {
                    const double sq = sqrt(disc);
                    eta = (a <= 0.0) ? (a - sq) / (2.0 * c) : 2.0 * b / (a + sq);
                    ok = true;
                }
            }
            if (!ok || !isfinite(eta) || f * eta >= 0.0) eta = -f / df;
            double nt = tau + eta;
            if (!(nt > lb && nt < ub)) nt = 0.5 * (lb + ub);
            if (nt == tau) break;
            tau = nt;
            if (ub - lb <= 2.0 * TR_EPS * fmax(fabs(lb), fabs(ub))) break;
        }
    }
    const double dorg = sdl[org];
    for (int i = lane; i < k; i += 32) Drow[i] = (sdl[i] - dorg) - tau;
    if (lane == 0) lam_out[(size_t)m * n + lo + j] = dorg + tau;
}

// Loewner formula: zhat_i = sign(w_i) sqrt(-Delta_ii prod_{j!=i} Delta_ji/(dl_i - dl_j))
// Block = 64 columns i x ZH_G row groups: group g multiplies up the factors of rows j = g (mod ZH_G) chunks, the
// partial products are combined through shared memory (the product over 1000 factors is a serial chain per
// thread; more threads per column is the only way to shorten it).
#define ZH_C 64
#define ZH_G 8
__global__ void __launch_bounds__(ZH_C * ZH_G)
dc_zhat_kernel(int n, int level, DcWs ws, const int* __restrict__ skip)
{
    __shared__ double s_part[ZH_G][ZH_C];
    const int m = blockIdx.z;
    if (skip && skip[m]) return;
    const int node = blockIdx.y;
    const int k = ws.nodek[(size_t)m * ws.nodes_max + node];
    if ((int)blockIdx.x * ZH_C >= k) return;
    const int ix = threadIdx.x & (ZH_C - 1), g = threadIdx.x / ZH_C;
    const int i = blockIdx.x * ZH_C + ix;
    const int lo = dc_bnd(n, level, node);
    const double* dl = ws.dl + (size_t)m * n + lo;
    const double* Dm = ws.U + (size_t)m * n * n + (size_t)lo * n + lo;
    double prod = 1.0;
    if (i < k) {
        const double di = dl[i];
        // numerators and denominators are multiplied up in chunks of 8 terms (each factor lies in [1e-16, 4] after
        // the normalisation of T, so a chunk cannot over/underflow) and divided once per chunk
        for (int j0 = 8 * g; j0 < k; j0 += 8 * ZH_G) {
            double num = 1.0, den = 1.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int jj = j0 + u;
                const bool use = (jj < k) && (jj != i);
                num *= use ? Dm[(size_t)jj * n + i] : 1.0;
                den *= use ? (di - dl[jj]) : 1.0;
            }
            prod *= num / den;
        }
    }
    s_part[g][ix] = prod;
    __syncthreads();
    if (g == 0 && i < k) {
        double p = Dm[(size_t)i * n + i];
#pragma unroll
        for (int q = 0; q < ZH_G; ++q) p *= s_part[q][ix];
        ws.zhat[(size_t)m * n + lo + i] = copysign(sqrt(-p), ws.wnd[(size_t)m * n + lo + i]);
    }
}

// U[j][i] = zhat_i / Delta[j][i], rows normalised (row j = eigenvector j of D + rho z z^T)
__global__ void __launch_bounds__(256)
dc_vectors_kernel(int n, int level, DcWs ws, const int* __restrict__ skip)
{
    const int m = blockIdx.z;
    if (skip && skip[m]) return;
    const int node = blockIdx.y;
    const int k = ws.nodek[(size_t)m * ws.nodes_max + node];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int j = blockIdx.x * 8 + wid;
    if (j >= k) return;
    const int lo = dc_bnd(n, level, node);
    const double* zh = ws.zhat + (size_t)m * n + lo;
    double* Drow = ws.U + (size_t)m * n * n + (size_t)(lo + j) * n + lo;
    double ss = 0.0;
    for (int i = lane; i < k; i += 32) {
        const double s = zh[i] / Drow[i];
        Drow[i] = s;
        ss = fma(s, s, ss);
    }
    ss = gg_warp_sum(ss);
    const double inv = rsqrt(ss);
    for (int i = lane; i < k; i += 32) Drow[i] *= inv;
}

// Qout[lo+j][lo+c] = sum_i U[j][i] Qin[ndrow_i][lo+c]   (j < k, c < N), 64x64 tiles, DMMA
#define DG_T 64
#define DG_KC 16
__global__ void __launch_bounds__(256)
dc_gemm_kernel(int n, int level, const double* __restrict__ Qin, double* __restrict__ Qout, DcWs ws,
               const int* __restrict__ skip)
{
    __shared__ double As[2][DG_T][DG_KC + 4];       // U tile   [j][i]
    __shared__ double Bs[2][DG_KC][DG_T + 4];       // Qin tile [i][c]
    const int m = blockIdx.z / (1 << level), node = blockIdx.z % (1 << level);
    if (skip && skip[m]) return;
    const int k = ws.nodek[(size_t)m * ws.nodes_max + node];
    const int lo = dc_bnd(n, level, node), hi = dc_bnd(n, level, node + 1);
    const int N = hi - lo;
    const int j0 = blockIdx.y * DG_T, c0 = blockIdx.x * DG_T;
    if (j0 >= k || c0 >= N) return;
    const double* Um = ws.U + (size_t)m * n * n + (size_t)lo * n + lo;
    const double* Qm = Qin + (size_t)m * n * n;
    const int* ndrow = ws.ndrow + (size_t)m * n + lo;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;
    const int wr = wid >> 1, wc = wid & 1;          // 4 x 2 warps, 16 x 32 outputs each
    // K list of this column tile: first child's columns / second child's columns / all poles for the one tile that
    // straddles the split (klist == nullptr: identity)
    const int n1 = dc_bnd(n, level + 1, 2 * node + 1) - lo;
    const int* klist = nullptr;
    int kk = k;
    if (c0 + DG_T <= n1) {
        klist = ws.lista + (size_t)m * n + lo;
        kk = ws.nodeka[((size_t)m * ws.nodes_max + node) * 2];
    } else if (c0 >= n1) {
        klist = ws.listb + (size_t)m * n + lo;
        kk = ws.nodeka[((size_t)m * ws.nodes_max + node) * 2 + 1];
    }
    const int nchunks = (kk + DG_KC - 1) / DG_KC;

    auto load_chunk = [&](int ch, int buf) {
        const int i0 = ch * DG_KC;
        for (int idx = tid; idx < DG_T * DG_KC; idx += 256) {
            const int jj = idx / DG_KC, ii = idx % DG_KC;
            double* dst = &As[buf][jj][ii];
            if (j0 + jj < k && i0 + ii < kk) {
                const int ip = klist ? klist[i0 + ii] : i0 + ii;
                gg_cp_async8(dst, Um + (size_t)(j0 + jj) * n + ip);
            } else *dst = 0.0;
        }
        for (int idx = tid; idx < DG_KC * DG_T; idx += 256) {
            const int ii = idx / DG_T, cc = idx % DG_T;
            double* dst = &Bs[buf][ii][cc];
            if (i0 + ii < kk && c0 + cc < N) {
                const int ip = klist ? klist[i0 + ii] : i0 + ii;
                gg_cp_async8(dst, Qm + (size_t)ndrow[ip] * n + lo + c0 + cc);
            } else *dst = 0.0;
        }
        gg_cp_commit();
    };

    double acc[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }
    load_chunk(0, 0);
    for (int ch = 0; ch < nchunks; ++ch) {
        if (ch + 1 < nchunks) { load_chunk(ch + 1, (ch + 1) & 1); gg_cp_wait<1>(); }
        else gg_cp_wait<0>();
        __syncthreads();
        const int buf = ch & 1;
#pragma unroll
        for (int k0 = 0; k0 < DG_KC; k0 += 4) {
            double fa[2], fb[4];
#pragma unroll
            for (int a = 0; a < 2; ++a) fa[a] = As[buf][(wr * 2 + a) * 8 + fr][k0 + fc];
#pragma unroll
            for (int b = 0; b < 4; ++b) fb[b] = Bs[buf][k0 + fc][(wc * 4 + b) * 8 + fr];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) gg_dmma(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
        }
        __syncthreads();
    }
    double* Qo = Qout + (size_t)m * n * n;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int jj = j0 + (wr * 2 + a) * 8 + fr;
        if (jj < k) {
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int cc = c0 + (wc * 4 + b) * 8 + 2 * fc;
                double* dst = Qo + (size_t)(lo + jj) * n + lo + cc;
                if (cc < N) dst[0] = acc[a][b][0];
                if (cc + 1 < N) dst[1] = acc[a][b][1];
            }
        }
    }
}

// =============================================================================================
// stage 3: back-transformation  Vt <- Vt Q_H^T  (compact WY panels of BT_NB reflectors)
// =============================================================================================
// T factor of panel b: H_{j0}...H_{j0+nb-1} = I - V T V^T (forward, columnwise; LAPACK dlarft)
__global__ void __launch_bounds__(256)
bt_larft_kernel(const double* __restrict__ Vh, const double* __restrict__ tau, int n, double* __restrict__ Tm,
                int npanels, const int* __restrict__ skip)
{
    __shared__ double Gs[BT_NB][BT_NB + 1];
    __shared__ double Ts[BT_NB][BT_NB + 1];
    const int m = blockIdx.y, pb = blockIdx.x;
    if (skip && skip[m]) return;
    const int j0 = pb * BT_NB;
    const double* V = Vh + (size_t)m * n * n;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // Gram of the panel's reflectors (rows of Vh), entries a <= b only
    for (int pr = wid; pr < BT_NB * BT_NB; pr += 8) {
        const int a = pr / BT_NB, b = pr % BT_NB;
        if (a > b) continue;
        const int ja = j0 + a, jb = j0 + b;
        double s = 0.0;
        if (ja < n - 1 && jb < n - 1) {
            const double* va = V + (size_t)ja * n;
            const double* vb = V + (size_t)jb * n;
            for (int i = jb + 1 + lane; i < n; i += 32) s = fma(va[i], vb[i], s);
        }
        s = gg_warp_sum(s);
        if (lane == 0) Gs[a][b] = s;
    }
    for (int idx = threadIdx.x; idx < BT_NB * BT_NB; idx += 256) Ts[idx / BT_NB][idx % BT_NB] = 0.0;
    __syncthreads();
    // column recurrence: T[0:i,i] = -tau_i T[0:i,0:i] G[0:i,i]
    for (int i = 0; i < BT_NB; ++i) {
        const int ji = j0 + i;
        const double ti = (ji < n - 1) ? tau[(size_t)m * n + ji] : 0.0;
        if (threadIdx.x < i) {
            const int r = threadIdx.x;
            double s = 0.0;
            for (int c = r; c < i; ++c) s = fma(Ts[r][c], Gs[c][i], s);
            Ts[r][i] = -ti * s;
        }
        if (threadIdx.x == 0) Ts[i][i] = ti;
        __syncthreads();
    }
    double* To = Tm + ((size_t)m * npanels + pb) * BT_NB * BT_NB;
    for (int idx = threadIdx.x; idx < BT_NB * BT_NB; idx += 256) To[idx] = Ts[idx / BT_NB][idx % BT_NB];
}

// Each CTA owns BT_R rows of Q (row-major, n columns) and applies all panels, last to first:
//   Y = Band V_b ; Y <- Y T_b^T ; Band <- Band - Y V_b^T
#define BT_KC 32
__global__ void __launch_bounds__(256, 5)
bt_apply_kernel(double* __restrict__ Q, const double* __restrict__ Vh, const double* __restrict__ Tm, int n,
                int npanels, const int* __restrict__ skip)
{
    __shared__ double Bt[BT_R][BT_KC + 4];       // band tile   [r][i]
    __shared__ double Vt_[BT_NB][BT_KC + 4];     // panel tile  [jj][i]
    __shared__ double Ys[BT_R][BT_NB + 4];
    __shared__ double Y2[BT_R][BT_NB + 4];
    __shared__ double Tsm[BT_NB][BT_NB + 1];
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    const int r0 = blockIdx.x * BT_R;
    double* Qm = Q + (size_t)m * n * n;
    const double* V = Vh + (size_t)m * n * n;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;
    // 4x4 output tiles of 8x8 over 8 warps: warp -> tile row (wid>>1), tile cols (wid&1)*2 + {0,1}
    const int tr = wid >> 1, tc0 = (wid & 1) * 2;

    for (int pb = npanels - 1; pb >= 0; --pb) {
        const int j0 = pb * BT_NB;
        const int istart = ((j0 + 1) / BT_KC) * BT_KC;        // reflectors of this panel vanish below j0+1
        const double* Tg = Tm + ((size_t)m * npanels + pb) * BT_NB * BT_NB;
        for (int idx = tid; idx < BT_NB * BT_NB; idx += 256) Tsm[idx / BT_NB][idx % BT_NB] = Tg[idx];
        // ---- Y = Band V_b ------------------------------------------------------------------
        // software pipeline: the next 32x32 band / panel tiles are fetched into registers while the
        // current ones (in shared memory) feed the tensor cores
        double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
        double pb_[4], pv_[4];
        auto fetch = [&](int i0, bool band) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int idx = tid + 256 * q;
                const int r = idx / BT_KC, ii = idx % BT_KC;
                const int gi = i0 + ii, gj = j0 + r, gr = r0 + r;
                pv_[q] = (gj < n - 1 && gi < n) ? V[(size_t)gj * n + gi] : 0.0;
                if (band) pb_[q] = (gr < n && gi < n) ? Qm[(size_t)gr * n + gi] : 0.0;
            }
        };
        auto stash = [&](bool band) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int idx = tid + 256 * q;
                const int r = idx / BT_KC, ii = idx % BT_KC;
                Vt_[r][ii] = pv_[q];
                if (band) Bt[r][ii] = pb_[q];
            }
        };
        fetch(istart, true);
        for (int i0 = istart; i0 < n; i0 += BT_KC) {
            stash(true);
            __syncthreads();
            if (i0 + BT_KC < n) fetch(i0 + BT_KC, true);
#pragma unroll
            for (int k0 = 0; k0 < BT_KC; k0 += 4) {
                const double fa = Bt[tr * 8 + fr][k0 + fc];
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const double fb = Vt_[(tc0 + b) * 8 + fr][k0 + fc];
                    gg_dmma(acc[b][0], acc[b][1], fa, fb);
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            Ys[tr * 8 + fr][(tc0 + b) * 8 + 2 * fc] = acc[b][0];
            Ys[tr * 8 + fr][(tc0 + b) * 8 + 2 * fc + 1] = acc[b][1];
        }
        __syncthreads();
        // ---- Y2 = Y T^T :  Y2[r][a] = sum_b Y[r][b] T[a][b]  (T upper triangular: b >= a) -------
        for (int idx = tid; idx < BT_R * BT_NB; idx += 256) {
            const int r = idx / BT_NB, a = idx % BT_NB;
            double s = 0.0;
            for (int b = a; b < BT_NB; ++b) s = fma(Ys[r][b], Tsm[a][b], s);
            Y2[r][a] = s;
        }
        __syncthreads();
        // ---- Band -= Y2 V_b^T -------------------------------------------------------------------
        fetch(istart, false);
        for (int i0 = istart; i0 < n; i0 += BT_KC) {
            stash(false);
            __syncthreads();
            if (i0 + BT_KC < n) fetch(i0 + BT_KC, false);
            // output tile: BT_R x BT_KC = 4 x 4 tiles of 8x8; warp -> row tile tr, col tiles tc0 + {0,1}
            double o[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
            for (int k0 = 0; k0 < BT_NB; k0 += 4) {
                const double fa = Y2[tr * 8 + fr][k0 + fc];
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const double fb = Vt_[k0 + fc][(tc0 + b) * 8 + fr];
                    gg_dmma(o[b][0], o[b][1], fa, fb);
                }
            }
            const int gr = r0 + tr * 8 + fr;
            if (gr < n) {
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int gi = i0 + (tc0 + b) * 8 + 2 * fc;
                    double* dst = Qm + (size_t)gr * n + gi;
                    if (gi < n) dst[0] -= o[b][0];
                    if (gi + 1 < n) dst[1] -= o[b][1];
                }
            }
            __syncthreads();
        }
    }
}

// ---- blocked back-transformation for larger n ---------------------------------------------------------------
// bt_apply_kernel walks 32-reflector panels; every panel re-reads the CTA's band of Vt twice and writes it once,
// which makes the stage L2-bandwidth bound (measured 25% of the DMMA peak).  For n >= BB_MIN the reflectors are
// grouped into blocks of BB_NB = 128 and each block is applied with two real GEMMs:
//     Vt <- Vt H_{j0+127} ... H_{j0} = Vt - (Vt V^T) (X V),      V = rows j0..j0+127 of Vh (128 x n)
// where X = T^T is the lower triangular matrix of the backward recurrence
//     w_i = tau_i ( y_i - sum_{q>i} w_q G_qi ),  G = V V^T  =>  X[a][i] = -tau_i sum_{q=i+1..a} X[a][q] G[q][i],  X[a][a] = tau_a.
// G, X and V' = X V do not depend on Vt and are formed for all blocks at once (three launches); the blocks are
// then applied last to first with Y = Vt V^T (bb_y_kernel) and Vt -= Y V' (bb_upd_kernel).  All five products run
// on the FP64 tensor cores through one 64x64-tile routine (cp.async double buffer, as dc_gemm_kernel).
#define BB_NB 128
#define BB_MIN 256
#define BB_T 64
#define BB_KC 16

struct BbSmem {
    double As[2][BB_T][BB_KC + 4];
    double Bs[2][BB_T * (BB_KC + 4)];            // NT: [c][k] stride KC+4 ; NN: [k][c] stride BB_T+4 (fits: 16*68 <= 64*20)
};

// acc += A[r0.., 0..K) * op(B): NT: op(B)[k][c] = B[c*ldb + k];  NN: op(B)[k][c] = B[k*ldb + c].
// Rows r >= Mr / columns c >= Nc / k >= K read as zero.  Fragment layout of gg_dmma (see gg_common.cuh).
template <bool TRANSB>
__device__ __forceinline__ void bb_gemm_tile(const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb,
                                             int Mr, int Nc, int K, int r0, int c0, double (&acc)[2][4][2], BbSmem& sm)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;
    const int wr = wid >> 1, wc = wid & 1;          // 4 x 2 warps, 16 x 32 outputs each
    const int nchunks = (K + BB_KC - 1) / BB_KC;
    auto load_chunk = [&](int ch, int buf) {
        const int k0 = ch * BB_KC;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int idx = tid + 256 * q;
            const int rr = idx / BB_KC, kk = idx % BB_KC;
            double* dst = &sm.As[buf][rr][kk];
            if (r0 + rr < Mr && k0 + kk < K) gg_cp_async8(dst, A + (size_t)(r0 + rr) * lda + k0 + kk);
            else *dst = 0.0;
        }
        if (TRANSB) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int idx = tid + 256 * q;
                const int cc = idx / BB_KC, kk = idx % BB_KC;
                double* dst = &sm.Bs[buf][cc * (BB_KC + 4) + kk];
                if (c0 + cc < Nc && k0 + kk < K) gg_cp_async8(dst, B + (size_t)(c0 + cc) * ldb + k0 + kk);
                else *dst = 0.0;
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int idx = tid + 256 * q;
                const int kk = idx / BB_T, cc = idx % BB_T;
                double* dst = &sm.Bs[buf][kk * (BB_T + 4) + cc];
                if (c0 + cc < Nc && k0 + kk < K) gg_cp_async8(dst, B + (size_t)(k0 + kk) * ldb + c0 + cc);
                else *dst = 0.0;
            }
        }
        gg_cp_commit();
    };
    load_chunk(0, 0);
    for (int ch = 0; ch < nchunks; ++ch) {
        if (ch + 1 < nchunks) { load_chunk(ch + 1, (ch + 1) & 1); gg_cp_wait<1>(); }
        else gg_cp_wait<0>();
        __syncthreads();
        const int buf = ch & 1;
#pragma unroll
        for (int k0 = 0; k0 < BB_KC; k0 += 4) {
            double fa[2], fb[4];
#pragma unroll
            for (int a = 0; a < 2; ++a) fa[a] = sm.As[buf][(wr * 2 + a) * 8 + fr][k0 + fc];
#pragma unroll
            for (int b = 0; b < 4; ++b)
                fb[b] = TRANSB ? sm.Bs[buf][((wc * 4 + b) * 8 + fr) * (BB_KC + 4) + k0 + fc]
                               : sm.Bs[buf][(k0 + fc) * (BB_T + 4) + (wc * 4 + b) * 8 + fr];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) gg_dmma(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
        }
        __syncthreads();
    }
}

// C[r][c] = acc (SUB: C[r][c] -= acc) for the 64x64 tile at (r0, c0), bounds Mr x Nc
template <bool SUB>
__device__ __forceinline__ void bb_store_tile(double* __restrict__ C, int ldc, int Mr, int Nc, int r0, int c0,
                                              const double (&acc)[2][4][2])
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int fr = lane >> 2, fc = lane & 3, wr = wid >> 1, wc = wid & 1;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int r = r0 + (wr * 2 + a) * 8 + fr;
        if (r < Mr) {
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int c = c0 + (wc * 4 + b) * 8 + 2 * fc;
                double* dst = C + (size_t)r * ldc + c;
                if (c < Nc) dst[0] = SUB ? dst[0] - acc[a][b][0] : acc[a][b][0];
                if (c + 1 < Nc) dst[1] = SUB ? dst[1] - acc[a][b][1] : acc[a][b][1];
            }
        }
    }
}

#define BB_ZERO_ACC(acc)                                                          \
    _Pragma("unroll") for (int a_ = 0; a_ < 2; ++a_)                                \
        _Pragma("unroll") for (int b_ = 0; b_ < 4; ++b_) { acc[a_][b_][0] = 0.0; acc[a_][b_][1] = 0.0; }

// G_P = V_P V_P^T for every block P of every matrix.  grid (2, 2, M*npb)
__global__ void __launch_bounds__(256)
bb_gram_kernel(const double* __restrict__ Vh, int n, int npb, double* __restrict__ G, const int* __restrict__ skip)
{
    __shared__ BbSmem sm;
    const int m = blockIdx.z / npb, P = blockIdx.z % npb;
    if (skip && skip[m]) return;
    const int j0 = P * BB_NB, i0 = j0 + 1;
    const int rows = min(BB_NB, n - j0);
    const double* V = Vh + (size_t)m * n * n + (size_t)j0 * n + i0;
    double acc[2][4][2];
    BB_ZERO_ACC(acc);
    bb_gemm_tile<true>(V, n, V, n, rows, rows, n - i0, blockIdx.y * BB_T, blockIdx.x * BB_T, acc, sm);
    bb_store_tile<false>(G + (size_t)blockIdx.z * BB_NB * BB_NB, BB_NB, BB_NB, BB_NB, blockIdx.y * BB_T, blockIdx.x * BB_T, acc);
}

// X_P (lower triangular, = T^T of the block): rows are independent; eight lanes share a row (they split the dot
// product of every recurrence step), four rows per warp.  grid (npb, M), 8 * BB_NB threads
// The strictly lower triangle of G is staged in shared memory first (packed rows, 65 KB): the 127 steps of the
// recurrence are strictly dependent, and reading G from global memory put an L2 round trip into every one of them
// (0.22 ms per eigh at K=20, p=1000 for 20 KFLOP of work per row).
#define BB_GTRI (BB_NB * (BB_NB - 1) / 2)
__device__ __forceinline__ int bb_goff(int i) { return i * (BB_NB - 1) - i * (i - 1) / 2; }   // row i: q = i+1..127
__global__ void __launch_bounds__(8 * BB_NB)
bb_x_kernel(const double* __restrict__ G, const double* __restrict__ tau, int n, int npb, double* __restrict__ X,
            const int* __restrict__ skip)
{
    extern __shared__ double xs[];                   // [BB_NB][BB_NB + 1], then gs[BB_GTRI]
    double* gs = xs + BB_NB * (BB_NB + 1);
    const int m = blockIdx.y, P = blockIdx.x;
    if (skip && skip[m]) return;
    const int j0 = P * BB_NB, a = threadIdx.x >> 3, l = threadIdx.x & 7;
    const int amax = a | 3;                          // last row handled by this warp
    const double* Gp = G + ((size_t)m * npb + P) * BB_NB * BB_NB;
    const double* tp = tau + (size_t)m * n + j0;
    for (int idx = threadIdx.x; idx < BB_NB * BB_NB; idx += 8 * BB_NB) {
        const int i = idx / BB_NB, q = idx % BB_NB;  // G is symmetric: row i, contiguous in q
        if (q > i) gs[bb_goff(i) + q - i - 1] = Gp[idx];
    }
    double* xr = xs + (size_t)a * (BB_NB + 1);
    for (int i = a + 1 + l; i < BB_NB; i += 8) xr[i] = 0.0;
    if (l == 0) xr[a] = (j0 + a < n - 1) ? tp[a] : 0.0;
    __syncthreads();
    for (int i = amax - 1; i >= 0; --i) {
        const double* gi = gs + bb_goff(i) - i - 1;  // gi[q] = G[i][q], q > i
        double sacc = 0.0;
        if (i < a)
            for (int q = i + 1 + l; q <= a; q += 8) sacc = fma(xr[q], gi[q], sacc);
        sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
        sacc += __shfl_xor_sync(0xffffffffu, sacc, 2);
        sacc += __shfl_xor_sync(0xffffffffu, sacc, 4);
        if (i < a && l == 0) xr[i] = -((j0 + i < n - 1) ? tp[i] : 0.0) * sacc;
        __syncwarp();
    }
    __syncthreads();
    double* Xp = X + ((size_t)m * npb + P) * BB_NB * BB_NB;
    for (int idx = threadIdx.x; idx < BB_NB * BB_NB; idx += 8 * BB_NB)
        Xp[idx] = xs[(size_t)(idx / BB_NB) * (BB_NB + 1) + idx % BB_NB];
}

// V'_P = X_P V_P  (rows j0..j0+127 of Vp, columns >= j0+1).  grid (ceil(n/64), 2, M*npb)
__global__ void __launch_bounds__(256)
bb_vprime_kernel(const double* __restrict__ Vh, const double* __restrict__ X, int n, int npb, double* __restrict__ Vp,
                 const int* __restrict__ skip)
{
    __shared__ BbSmem sm;
    const int m = blockIdx.z / npb, P = blockIdx.z % npb;
    if (skip && skip[m]) return;
    const int j0 = P * BB_NB, i0 = j0 + 1, len = n - i0;
    const int c0 = blockIdx.x * BB_T, r0 = blockIdx.y * BB_T;
    if (c0 >= len) return;
    const int rows = min(BB_NB, n - j0);
    double acc[2][4][2];
    BB_ZERO_ACC(acc);
    bb_gemm_tile<false>(X + (size_t)blockIdx.z * BB_NB * BB_NB, BB_NB, Vh + (size_t)m * n * n + (size_t)j0 * n + i0, n,
                        rows, len, rows, r0, c0, acc, sm);
    bb_store_tile<false>(Vp + (size_t)m * n * n + (size_t)j0 * n + i0, n, rows, len, r0, c0, acc);
}

// Y = Vt[:, i0:] V_P^T   (n x 128).  grid (2, ceil(n/64), M)
__global__ void __launch_bounds__(256)
bb_y_kernel(const double* __restrict__ Q, const double* __restrict__ Vh, int n, int P, double* __restrict__ Y,
            const int* __restrict__ skip)
{
    __shared__ BbSmem sm;
    const int m = blockIdx.z;
    if (skip && skip[m]) return;
    const int j0 = P * BB_NB, i0 = j0 + 1;
    const int rows = min(BB_NB, n - j0);
    double acc[2][4][2];
    BB_ZERO_ACC(acc);
    bb_gemm_tile<true>(Q + (size_t)m * n * n + i0, n, Vh + (size_t)m * n * n + (size_t)j0 * n + i0, n,
                       n, rows, n - i0, blockIdx.y * BB_T, blockIdx.x * BB_T, acc, sm);
    bb_store_tile<false>(Y + (size_t)m * n * BB_NB, BB_NB, n, BB_NB, blockIdx.y * BB_T, blockIdx.x * BB_T, acc);
}

// Vt[:, i0:] -= Y V'_P.  grid (ceil(len/64), ceil(n/64), M)
__global__ void __launch_bounds__(256)
bb_upd_kernel(double* __restrict__ Q, const double* __restrict__ Vp, const double* __restrict__ Y, int n, int P,
              const int* __restrict__ skip)
{
    __shared__ BbSmem sm;
    const int m = blockIdx.z;
    if (skip && skip[m]) return;
    const int j0 = P * BB_NB, i0 = j0 + 1, len = n - i0;
    const int rows = min(BB_NB, n - j0);
    double acc[2][4][2];
    BB_ZERO_ACC(acc);
    bb_gemm_tile<false>(Y + (size_t)m * n * BB_NB, BB_NB, Vp + (size_t)m * n * n + (size_t)j0 * n + i0, n,
                        n, len, rows, blockIdx.y * BB_T, blockIdx.x * BB_T, acc, sm);
    bb_store_tile<true>(Q + (size_t)m * n * n + i0, n, n, len, blockIdx.y * BB_T, blockIdx.x * BB_T, acc);
}

// ---- small helpers ----------------------------------------------------------------------------
__global__ void tr_skip_kernel(const double* __restrict__ ctrl, int mpp, int M, int* __restrict__ skip)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < M) skip[m] = (ctrl && ctrl[(size_t)(m / mpp) * GG_CTRL_STRIDE + GG_C_DONE] != 0.0) ? 1 : 0;
}

__global__ void tr_copy_rows_kernel(const double* __restrict__ src, double* __restrict__ dst, size_t per, const int* skip)
{
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < per; e += (size_t)gridDim.x * blockDim.x)
        dst[(size_t)m * per + e] = src[(size_t)m * per + e];
}

__global__ void tr_zero_kernel(double* __restrict__ dst, size_t per, const int* skip)
{
    const int m = blockIdx.y;
    if (skip && skip[m]) return;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < per; e += (size_t)gridDim.x * blockDim.x)
        dst[(size_t)m * per + e] = 0.0;
}

// =============================================================================================
// host driver
// =============================================================================================
static inline size_t al(size_t x) { return (x + 255) / 256 * 256; }

static int dc_levels(int n)
{
    int L = 0;
    while (((n + (1 << L) - 1) >> L) > DC_LEAF) ++L;
    return L;
}

// diagnostics (GG_DEBUG_STAGE=1): synchronise and test an (M,n) array for non-finite entries on the host
static int dbg_nonfinite(const double* dptr, int M, int n, int ncheck, cudaStream_t s)
{
    std::vector<double> h((size_t)M * n);
    if (cudaMemcpyAsync(h.data(), dptr, sizeof(double) * M * n, cudaMemcpyDeviceToHost, s) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(s) != cudaSuccess) return 1;
    for (int m = 0; m < M; ++m)
        for (int i = 0; i < ncheck; ++i)
            if (!std::isfinite(h[(size_t)m * n + i])) return 1;
    return 0;
}

// Side streams for work forked off the caller's stream.  They and their events belong to the calling host thread and
// the current device (thread_local, created on first use), so concurrent solves on other host threads never share a
// stream or an event with this one.  Fork and join are event record / wait only, which is legal inside stream capture.
#define GG_SIDE_MAX 3
struct GgSides {
    cudaStream_t s[GG_SIDE_MAX];
    cudaEvent_t fork, join[GG_SIDE_MAX];
};

static GgSides* gg_sides()          // nullptr if they cannot be created
{
    static thread_local GgSides tl[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    GgSides& g = tl[dev];
    if (!g.fork && cudaEventCreateWithFlags(&g.fork, cudaEventDisableTiming) != cudaSuccess) {
        g.fork = nullptr;
        return nullptr;
    }
    for (int i = 0; i < GG_SIDE_MAX; ++i) {
        if (!g.s[i] && cudaStreamCreateWithFlags(&g.s[i], cudaStreamNonBlocking) != cudaSuccess) {
            g.s[i] = nullptr;
            return nullptr;
        }
        if (!g.join[i] && cudaEventCreateWithFlags(&g.join[i], cudaEventDisableTiming) != cudaSuccess) {
            g.join[i] = nullptr;
            return nullptr;
        }
    }
    return &g;
}

// side streams 0..k-1 wait for the work issued to s so far
static int gg_fork(const GgSides& g, cudaStream_t s, int k)
{
    cudaError_t e = cudaEventRecord(g.fork, s);
    for (int i = 0; i < k && e == cudaSuccess; ++i) e = cudaStreamWaitEvent(g.s[i], g.fork, 0);
    return (int)e;
}

// s waits for the work issued to side streams 0..k-1 so far (all k are joined even if one fails)
static int gg_join(const GgSides& g, cudaStream_t s, int k)
{
    cudaError_t r = cudaSuccess;
    for (int i = 0; i < k; ++i) {
        cudaError_t e = cudaEventRecord(g.join[i], g.s[i]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s, g.join[i], 0);
        if (r == cudaSuccess) r = e;
    }
    return (int)r;
}

// stage-1 workspace of matrices m0.. of the batch (every array has the matrix index outermost)
static TrWs tr_ws_from(const TrWs& tw, int m0, int n)
{
    const size_t nn = (size_t)n * n, mn = (size_t)m0 * n;
    TrWs t = tw;
    t.Vh += m0 * nn;
    t.tau += mn;
    t.d += mn;
    t.e += mn;
    t.vbuf += 2 * mn;
    t.w += TR_QMAX * mn;
    t.y += mn;
    t.cnt += m0;
#ifdef TR_TIMING
    if (m0) t.dbg = nullptr;         // only the chain that holds matrix 0 stamps
#endif
    return t;
}

// Concurrent chains of stage 1 (see gg_eigh_tridiag_impl): TR_GROUPS chains while the batch's upper triangles
// (4 M t^2 bytes) exceed TR_SPLIT_MB.  Measured on B200 (profiles/r03_tr_groups.json): two groups beat three and four,
// and 12 MB beats 6 / 24 / 48 MB (a lower threshold splits K=3 p=1000 and K=10 p=500, which then get slower).
#ifndef TR_GROUPS
#define TR_GROUPS 2
#endif
#ifndef TR_SPLIT_MB
#define TR_SPLIT_MB 12
#endif
static_assert(TR_GROUPS >= 1 && TR_GROUPS <= GG_SIDE_MAX + 1, "TR_GROUPS chains need TR_GROUPS - 1 side streams");

// write-back depth of the tridiagonalisation (see TR_QMAX): env GG_TR_LAZY in [1, TR_QMAX], default 3
int gg_tr_lazy_depth()
{
    static int q = -1;
    if (q < 0) {
        const char* ev = getenv("GG_TR_LAZY");
        q = ev ? atoi(ev) : 3;
        if (q < 1) q = 1;
        if (q > TR_QMAX) q = TR_QMAX;
    }
    return q;
}

size_t gg_tridiag_ws_bytes(int M, int n)
{
    const size_t nn = (size_t)n * n, Mn = (size_t)M * n;
    const int L = dc_levels(n);
    const int npanels = (n - 1 + BT_NB - 1) / BT_NB + 1;
    size_t b = 0;
    b += 3 * al(sizeof(double) * M * nn);                 // Vh, Q0, U
    b += 12 * al(sizeof(double) * Mn);                    // tau d e vbuf(2) w y lam0 lam1 z dl wnd zhat (13) -> see below
    b += (2 + TR_QMAX) * al(sizeof(double) * Mn);
    b += 3 * al(sizeof(int) * Mn) + 2 * al(sizeof(double) * Mn);   // ndrow, rotp, rotn, rotc, rots
    b += al(sizeof(int) * (size_t)M * (1 << L));          // nodek
    b += al(sizeof(int) * (size_t)M * (1 << L) * 2) + 2 * al(sizeof(int) * Mn);   // nodeka, lista, listb
    b += al(sizeof(int) * Mn) + al(sizeof(int) * (size_t)M * (1 << L));           // dfl, nodendf
    b += al(sizeof(double) * (size_t)M * (1 << L));       // noderho
    b += al(sizeof(double) * (size_t)M * npanels * BT_NB * BT_NB);
    b += 2 * al(sizeof(int) * (size_t)M);                 // skip, cnt
    b += al(sizeof(double) * (size_t)M);                  // scale
    b += 2 * al(sizeof(double) * (size_t)M * ((n + BB_NB - 1) / BB_NB) * BB_NB * BB_NB);   // G, X of the blocked back-transformation
    if (n >= BB_MIN) b += al(sizeof(double) * M * nn);   // V' = X V
    b += al(sizeof(double) * sytrd_blocked_ws_doubles(M, n));   // W panel of the blocked tridiagonalisation
    return b;
}

// mode bits for debugging/tests: stop_after 1 = after sytrd (A holds junk; outputs d,e in D/ws), 0 = full
int gg_eigh_tridiag_impl(double* A, double* D, int M, int n, const double* ctrl, int mpp, void* wsp, size_t ws_bytes,
                         cudaStream_t s, int which)
{
    if (ws_bytes < gg_tridiag_ws_bytes(M, n)) return -3;
    const size_t nn = (size_t)n * n, Mn = (size_t)M * n;
    const int L = dc_levels(n);
    const int npanels = (n - 1 + BT_NB - 1) / BT_NB;
    char* p = (char*)wsp;
    auto take = [&](size_t bytes) { char* r = p; p += al(bytes); return r; };
    TrWs tw;
    DcWs dw;
    tw.Vh = (double*)take(sizeof(double) * M * nn);
    double* Q0 = (double*)take(sizeof(double) * M * nn);
    dw.U = (double*)take(sizeof(double) * M * nn);
    tw.tau = (double*)take(sizeof(double) * Mn);
    tw.d = (double*)take(sizeof(double) * Mn);
    tw.e = (double*)take(sizeof(double) * Mn);
    tw.vbuf = (double*)take(sizeof(double) * 2 * Mn);
    tw.w = (double*)take(sizeof(double) * TR_QMAX * Mn);
    tw.y = (double*)take(sizeof(double) * Mn);
    dw.lam[0] = (double*)take(sizeof(double) * Mn);
    dw.lam[1] = (double*)take(sizeof(double) * Mn);
    dw.z = (double*)take(sizeof(double) * Mn);
    dw.dl = (double*)take(sizeof(double) * Mn);
    dw.wnd = (double*)take(sizeof(double) * Mn);
    dw.zhat = (double*)take(sizeof(double) * Mn);
    dw.ndrow = (int*)take(sizeof(int) * Mn);
    dw.rotc = (double*)take(sizeof(double) * Mn);
    dw.rots = (double*)take(sizeof(double) * Mn);
    dw.rotp = (int*)take(sizeof(int) * Mn);
    dw.rotn = (int*)take(sizeof(int) * Mn);
    dw.nodes_max = 1 << L;
    dw.nodek = (int*)take(sizeof(int) * (size_t)M * dw.nodes_max);
    dw.noderho = (double*)take(sizeof(double) * (size_t)M * dw.nodes_max);
    dw.nodeka = (int*)take(sizeof(int) * (size_t)M * dw.nodes_max * 2);
    dw.lista = (int*)take(sizeof(int) * Mn);
    dw.listb = (int*)take(sizeof(int) * Mn);
    dw.dfl = (int*)take(sizeof(int) * Mn);
    dw.nodendf = (int*)take(sizeof(int) * (size_t)M * dw.nodes_max);
    double* Tm = (double*)take(sizeof(double) * (size_t)M * (npanels + 1) * BT_NB * BT_NB);
    int* skip = (int*)take(sizeof(int) * (size_t)M);
    tw.cnt = (int*)take(sizeof(int) * (size_t)M);
    double* scale = (double*)take(sizeof(double) * (size_t)M);
    const int npb = (n - 1 + BB_NB - 1) / BB_NB;
    double* Gb = (double*)take(sizeof(double) * (size_t)M * ((n + BB_NB - 1) / BB_NB) * BB_NB * BB_NB);
    double* Xb = (double*)take(sizeof(double) * (size_t)M * ((n + BB_NB - 1) / BB_NB) * BB_NB * BB_NB);
    double* Vp = (n >= BB_MIN) ? (double*)take(sizeof(double) * M * nn) : nullptr;
    double* Wpanel = (double*)take(sizeof(double) * sytrd_blocked_ws_doubles(M, n));
    static int stop_after = -1;
    if (stop_after < 0) { const char* ev = getenv("GG_TR_STOP"); stop_after = ev ? atoi(ev) : 0; }

#ifdef TR_TIMING
    tw.dbg = (long long*)dw.U;            // U is not used before stage 2; read back by the timing script
#endif
    gg_count_launch(1);
    tr_skip_kernel<<<(M + 127) / 128, 128, 0, s>>>(ctrl, mpp, M, skip);
    GG_CHECK_LAUNCH();
    dim3 gz(64, M);
    gg_count_launch(1);
    tr_zero_kernel<<<gz, 256, 0, s>>>(tw.Vh, nn, skip);
    gg_count_launch(1);
    tr_zero_kernel<<<gz, 256, 0, s>>>(Q0, nn, skip);
    gg_count_launch(1);
    tr_zero_kernel<<<dim3(1, M), 256, 0, s>>>(tw.tau, (size_t)n, skip);
    GG_CHECK_LAUNCH();

    // ---- stage 1 ----
    {
        // the 2p-1 launches of this chain are short and strictly dependent: programmatic dependent launch
        // lets launch k+1 be set up while launch k drains (kernels start with griddepcontrol.wait)
        cudaLaunchAttribute pdl[1];
        pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        pdl[0].val.programmaticStreamSerializationAllowed = 1;
        cudaLaunchConfig_t cfg = {};
        cfg.stream = s;
        cfg.attrs = pdl;
        static int no_pdl = -1;
        if (no_pdl < 0) { const char* ev = getenv("GG_NO_PDL"); no_pdl = ev ? atoi(ev) : 0; }
        cfg.numAttrs = no_pdl ? 0 : 1;
        static int tr_old = -1;
        if (tr_old < 0) { const char* ev = getenv("GG_TR_OLD"); tr_old = ev ? atoi(ev) : 0; }
        // Stage 1 runs in up to three parts:
        //   columns [0, jb)   blocked path (cluster panel kernel + DMMA rank-2k update, gg_sytrd_blocked.cuh);
        //   columns [jb, js)  per-column chain (tr_col_kernel + tr_symv_kernel);
        //   columns [js, n)   shared-memory tail.
        // Measured on B200 (profiles/r02_sytrd_paths.json): at every batch shape tried the chain is as fast as or
        // faster than the blocked path (K=20, p=1000: 11.6 vs 11.9 ms; K=2, p=1000: 5.4 vs 7.2 ms), so jb = 0 by
        // default.  GG_TR_BLOCKED=1 uses the blocked path for every column below the tail, GG_TR_SWITCH_MB=x while
        // the batch's upper triangles (4 M t^2 bytes) exceed x MB; GG_TR_OLD=1 disables it.
        const int js_full = n > TR_TAIL ? n - TR_TAIL : 0;
        const bool prof12 = (which == 1 || which == 2);
        int jb = 0;
        if (!tr_old && n > TR_TAIL && n <= PB_NMAX) {
            const int nbp = sytrd_blocked_env("GG_TR_NB", 16) == 32 ? 32 : 16;
            const double sw = (double)sytrd_blocked_env("GG_TR_SWITCH_MB", 1 << 20) * 1048576.0;
            const bool all = sytrd_blocked_env("GG_TR_BLOCKED", 0) != 0;
            while (jb < js_full && (all || 4.0 * M * (double)(n - jb - 1) * (n - jb - 1) > sw)) jb += nbp;
            if (jb > js_full) jb = js_full;
        }
        const bool use_blocked = jb > 0;
        // profiling variants: with a blocked part, which = 1 / 2 time its panel kernels / rank-2k updates alone;
        // without one they time the column kernels / trailing-matrix passes of the chain over all columns (as before)
        const int js = (prof12 && !use_blocked) ? n : js_full;       // the tail takes over at column js
        if (use_blocked) {
            const int rc = sytrd_blocked_run(A, n, M, jb, tw, Wpanel, skip, s, prof12 ? which : 0);
            if (rc != 0) return rc;
            if (jb < js && !prof12) {
                // hand-over to the chain: nothing is pending, so the column kernel must find y = 0 (it then forms
                // w_{jb-1} = 0) and a finite previous vector
                tr_zero_kernel<<<dim3(1, M), 256, 0, s>>>(tw.y, (size_t)n, skip);
                tr_zero_kernel<<<dim3(2, M), 256, 0, s>>>(tw.vbuf, (size_t)2 * n, skip);
                gg_count_launch(2);
            }
        }
        const bool chain = !(use_blocked && prof12) && jb < js;
        const int lazy_q = gg_tr_lazy_depth();
        int kb = jb;                                  // pairs kb..j-1 are pending at step j
        // merged chain (GG_TR_MERGE=1, n - jb <= 2048): column step jb alone, then one tr_step_kernel per column.
        // Measured on B200 (profiles/r02_chain_merge.json) it is SLOWER than the two-launch chain at every shape
        // (K=20 p=1000: 13.4 vs 12.0 ms, K=3: 6.1 vs 5.7, K=10 p=500: 2.85 vs 2.58): the arrival counter + acquire +
        // re-read of y through L2 costs more than a programmatic-dependent-launch boundary, and the grid after a
        // write pass loses its early tile loads.  Kept as an option, not the default.
        const int tr_merge = sytrd_blocked_env("GG_TR_MERGE", 0);
        const bool merged = tr_merge && chain && !prof12 && (n - jb) <= 2048 && js > jb && js < n;
        if (merged) {
            if (cudaMemsetAsync(tw.cnt, 0, sizeof(int) * (size_t)M, s) != cudaSuccess) return -6;
            int prev_write = 1;                       // (nothing is in flight before the first step: either is safe)
            for (int j = jb; j < js; ++j) {
                if (j == jb) {
                    const int len = n - j;
                    cfg.gridDim = dim3(M); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0;
                    cudaError_t e;
                    gg_count_launch(1);
                    if (len <= 512) e = cudaLaunchKernelEx(&cfg, tr_col_kernel<2, 256, true>, (const double*)A, n, j, kb, tw, (const int*)skip);
                    else if (len <= 1024) e = cudaLaunchKernelEx(&cfg, tr_col_kernel<4, 256, true>, (const double*)A, n, j, kb, tw, (const int*)skip);
                    else e = cudaLaunchKernelEx(&cfg, tr_col_kernel<8, 256, true>, (const double*)A, n, j, kb, tw, (const int*)skip);
                    if (e != cudaSuccess) return (int)e;
                }
                const int write = (j - kb >= lazy_q || (j == js - 1 && j > kb)) ? 1 : 0;
                const int t = n - j - 1;
                const int nt = (t + SV_T - 1) / SV_T;
                cfg.gridDim = dim3(nt * (nt + 1) / 2, M); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0;
                gg_count_launch(1);
                // the grid after the standalone column kernel must not load early either: that kernel releases its
                // dependents after ITS wait, but the grid before it may be a blocked-path kernel without the protocol
                cudaError_t e = cudaLaunchKernelEx(&cfg, tr_step_kernel, A, n, j, kb, write, tw, (const int*)skip, nt,
                                                   (prev_write || j == jb) ? 0 : 1, (j + 1 < js) ? 1 : 0);
                if (e != cudaSuccess) return (int)e;
                prev_write = write;
                if (write) kb = j;
            }
        }
        // Attributes of a chain launch: programmatic dependence on the stream's previous kernel unless `dep` is false
        // (the first launch after a fork or a join, which must wait for the event in full); with `prio` the greatest
        // scheduling priority (see the concurrent chains below).
        int prio_lo = 0, prio_hi = 0;
        cudaLaunchAttribute ca[2];
        auto chain_cfg = [&](cudaStream_t st, bool dep, bool prio) {
            cfg.stream = st;
            cfg.attrs = ca;
            cfg.numAttrs = 0;
            if (dep && !no_pdl) {
                ca[cfg.numAttrs].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                ca[cfg.numAttrs++].val.programmaticStreamSerializationAllowed = 1;
            }
            if (prio) {
                ca[cfg.numAttrs].id = cudaLaunchAttributePriority;
                ca[cfg.numAttrs++].val.priority = prio_hi;
            }
        };
        // column step j and trailing-matrix pass j over the Mb matrices of (Ab, twb, skb), on stream st
        auto column = [&](double* Ab, const TrWs& twb, const int* skb, int Mb, cudaStream_t st, bool dep, bool prio,
                          int j, int write) -> int {
            if (which != 2) {
                const int len = n - j;
                const int thr = len <= 2048 ? 256 : 512;
                chain_cfg(st, dep, prio);
                cfg.gridDim = dim3(Mb); cfg.blockDim = dim3(thr); cfg.dynamicSmemBytes = 0;
                cudaError_t e;
                gg_count_launch(1);
                if (len <= 512) e = cudaLaunchKernelEx(&cfg, tr_col_kernel<2, 256, true>, (const double*)Ab, n, j, kb, twb, skb);
                else if (len <= 1024) e = cudaLaunchKernelEx(&cfg, tr_col_kernel<4, 256, true>, (const double*)Ab, n, j, kb, twb, skb);
                else if (len <= 2048) e = cudaLaunchKernelEx(&cfg, tr_col_kernel<8, 256, true>, (const double*)Ab, n, j, kb, twb, skb);
                else if (len <= 8192) e = cudaLaunchKernelEx(&cfg, tr_col_kernel<16, 512, false>, (const double*)Ab, n, j, kb, twb, skb);
                else return -5;
                if (e != cudaSuccess) return (int)e;
                dep = true;
            }
            if (j < n - 1 && which != 1) {
                const int t = n - j - 1;
                const int nt = (t + SV_T - 1) / SV_T;
                chain_cfg(st, dep, false);
                cfg.gridDim = dim3(nt * (nt + 1) / 2, Mb); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0;
                gg_count_launch(1);
                cudaError_t e = cudaLaunchKernelEx(&cfg, tr_symv_kernel, Ab, n, j, kb, write, twb, skb, nt);
                if (e != cudaSuccess) return (int)e;
            }
            return 0;
        };
        // write pass: the pending list is full, or the tail kernel takes over next (it expects only pair js-1)
        auto write_pass = [&](int j) { return (j - kb >= lazy_q || (j == js - 1 && j > kb)) ? 1 : 0; };

        // Columns [jb, jg): concurrent chains.  The chain is serial only within a matrix (y_j -> v_j -> y_{j+1}), so
        // while the trailing blocks are large the batch runs as G chains over contiguous groups of matrices, group g
        // on side stream g-1 (group 0 on s): one chain's column step and launch boundaries overlap another's
        // trailing-matrix pass, whose tiles also fill the last, partial wave of the other grids.  Launches are issued
        // column-major, so every chain is at the same column with the same write-back schedule kb, and the chains
        // rejoin at column jg to go on as one chain over the batch: short columns cannot afford G times the host
        // time of their launches (about 2 us each).  The column steps run at the greatest scheduling priority: they
        // are on their chain's critical path, and their CTAs must not queue behind the pending tiles of another
        // chain's pass (measured at K=20, p=1000 with a 24 MB threshold: gg_eigh 15.19 ms with, 15.86 ms without).
        const int G = M < TR_GROUPS ? M : TR_GROUPS;
        int jg = jb;
        GgSides* sides = nullptr;
        if (chain && !merged && !use_blocked && G > 1) {
            while (jg < js && 4.0 * M * (double)(n - jg - 1) * (n - jg - 1) > TR_SPLIT_MB * 1048576.0) ++jg;
            if (jg > jb && (!(sides = gg_sides()) || gg_fork(*sides, s, G - 1) != 0)) jg = jb;
            if (jg > jb) cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        }
        bool dep = true;                  // the next launch on s may depend programmatically on its predecessor
        if (jg > jb) {
            TrWs twg[TR_GROUPS];
            for (int g = 0; g < G; ++g) twg[g] = tr_ws_from(tw, g * M / G, n);
            int rc = 0;
            for (int j = jb; j < jg && rc == 0; ++j) {
                const int write = write_pass(j);
                for (int g = 0; g < G && rc == 0; ++g) {
                    const int m0 = g * M / G, m1 = (g + 1) * M / G;
                    rc = column(A + m0 * nn, twg[g], skip + m0, m1 - m0, g ? sides->s[g - 1] : s, j > jb, true, j,
                                write);
                }
                if (write) kb = j;
            }
            const int rj = gg_join(*sides, s, G - 1);
            if (rc != 0) return rc;
            if (rj != 0) return rj;
            dep = false;
        }
        for (int j = jg; j < js && chain && !merged; ++j) {
            const int write = write_pass(j);
            const int rc = column(A, tw, skip, M, s, dep, false, j, write);
            if (rc != 0) return rc;
            dep = true;
            if (write) kb = j;
        }
        if (js < n && !(use_blocked && prof12)) {
            const int ts = n - js;
            const size_t tsm = sizeof(double) * ((size_t)ts * (ts | 1) + 3 * ts + 64 + 4);
            cudaFuncSetAttribute(tr_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,       // (per device)
                                 (int)(sizeof(double) * ((size_t)TR_TAIL * (TR_TAIL | 1) + 3 * TR_TAIL + 68)));
            chain_cfg(s, dep, false);
            cfg.gridDim = dim3(M); cfg.blockDim = dim3(512); cfg.dynamicSmemBytes = tsm;
            gg_count_launch(1);
            cudaError_t e = cudaLaunchKernelEx(&cfg, tr_tail_kernel, (const double*)A, n, js, tw, (const int*)skip, chain ? 1 : 0);
            if (e != cudaSuccess) return (int)e;
        }
    }
    GG_CHECK_LAUNCH();
    static int dbg_stage = -1;
    if (dbg_stage < 0) { const char* ev = getenv("GG_DEBUG_STAGE"); dbg_stage = ev ? atoi(ev) : 0; }
    if (dbg_stage && (which == 0 || which == 4)) {
        if (dbg_nonfinite(tw.d, M, n, n, s)) return -11;
        if (dbg_nonfinite(tw.e, M, n, n - 1, s)) return -12;
        if (dbg_nonfinite(tw.tau, M, n, n - 1, s)) return -13;
    }
    if (stop_after == 1 || (which != 0 && which != 4)) return 0;

    // ---- stage 3 preparation: G, X, V' of the blocked back-transformation (independent of stage 2).
    // (Round 1: running these three launches on a side stream next to the divide & conquer kernels gained 0.3 ms at
    // cfg3 but corrupted results when five host threads drove five solves concurrently -- DESIGN.md 4.4.  The
    // GG_BT_SIDE=1 variant below shares nothing between threads and passed the concurrent-solve stress test, but
    // since the round-1 failure was never explained the default stays: plain launches on the caller's stream.)
    static int bt_big = -1;
    if (bt_big < 0) {
        const char* ev = getenv("GG_BT_BIG");
        bt_big = ev ? atoi(ev) : 1;
    }
    cudaFuncSetAttribute(bb_x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,                  // (per device)
                         (int)(sizeof(double) * (BB_NB * (BB_NB + 1) + BB_GTRI)));
    const bool use_big = npanels > 0 && which != 4 && bt_big && n >= BB_MIN;
    // GG_BT_SIDE=1: the three preparation launches run on side stream 0 of the calling thread (gg_sides) next to
    // stage 2 (fork after stage 1, join before stage 3): nothing is shared between concurrent solves.
    GgSides* bt_side = nullptr;
    if (use_big) {
        cudaStream_t ps = s;
        if (sytrd_blocked_env("GG_BT_SIDE", 0) && (bt_side = gg_sides()) && gg_fork(*bt_side, s, 1) == 0)
            ps = bt_side->s[0];
        else
            bt_side = nullptr;
        const int nt64 = (n + BB_T - 1) / BB_T;
        gg_count_launch(1);
        bb_gram_kernel<<<dim3(BB_NB / BB_T, BB_NB / BB_T, M * npb), 256, 0, ps>>>(tw.Vh, n, npb, Gb, skip);
        gg_count_launch(1);
        bb_x_kernel<<<dim3(npb, M), 8 * BB_NB, sizeof(double) * (BB_NB * (BB_NB + 1) + BB_GTRI), ps>>>(Gb, tw.tau, n, npb, Xb, skip);
        gg_count_launch(1);
        bb_vprime_kernel<<<dim3(nt64, BB_NB / BB_T, M * npb), 256, 0, ps>>>(tw.Vh, Xb, n, npb, Vp, skip);
        GG_CHECK_LAUNCH();
    }

    // ---- stage 2 ----
    // buffers: leaves write Qt into buf[L & 1 ? ...]; arrange so that the root lands in A.
    double* qbuf[2] = {A, Q0};           // level l merge reads qbuf[(l+1)&1], writes qbuf[l&1]; root (l=0) -> A
    gg_count_launch(1);
    tr_zero_kernel<<<gz, 256, 0, s>>>(A, nn, skip);
    gg_count_launch(1);
    dc_scale_kernel<<<M, 256, 0, s>>>(tw.d, tw.e, n, scale, skip);
    if (L > 0) {
        const int nsplit = (1 << L) - 1;
        gg_count_launch(1);
        dc_tear_kernel<<<dim3((nsplit + 127) / 128, M), 128, 0, s>>>(tw.d, tw.e, n, L, skip);
    }
    gg_count_launch(1);
    dc_leaf_kernel<<<dim3(1 << L, M), 128, 0, s>>>(tw.d, tw.e, n, L, dw.lam[L & 1], qbuf[L & 1], skip);
    GG_CHECK_LAUNCH();
    if (dbg_stage && dbg_nonfinite(dw.lam[L & 1], M, n, n, s)) return -14;
    {
        cudaFuncSetAttribute(dc_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);   // (per device)
        cudaFuncSetAttribute(dc_secular_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    }
    for (int l = L - 1; l >= 0; --l) {
        const int nodes = 1 << l;
        const int Nmax = ((n + nodes - 1) >> l) + 1;
        const size_t psm = sizeof(double) * 2 * Nmax + sizeof(int) * 3 * Nmax + Nmax + 16;
        if (psm > 200 * 1024) return -4;
        const double* Qin = qbuf[(l + 1) & 1];
        double* Qout = qbuf[l & 1];
        gg_count_launch(1);
        dc_prepare_kernel<<<dim3(nodes, M), 1024, psm, s>>>(tw.e, n, l, dw.lam[(l + 1) & 1], dw.lam[l & 1],
                                                            (double*)Qin, Qout, dw, skip);
        gg_count_launch(1);
        dc_copy_deflated_kernel<<<dim3((Nmax + 7) / 8, nodes, M), 256, 0, s>>>(n, l, Qin, Qout, dw, skip);
        gg_count_launch(1);
        dc_secular_kernel<<<dim3((Nmax + 7) / 8, nodes, M), 256, sizeof(double) * 2 * Nmax, s>>>(n, l, dw.lam[l & 1], dw, skip);
        gg_count_launch(1);
        dc_zhat_kernel<<<dim3((Nmax + ZH_C - 1) / ZH_C, nodes, M), ZH_C * ZH_G, 0, s>>>(n, l, dw, skip);
        gg_count_launch(1);
        dc_vectors_kernel<<<dim3((Nmax + 7) / 8, nodes, M), 256, 0, s>>>(n, l, dw, skip);
        gg_count_launch(1);
        dc_gemm_kernel<<<dim3((Nmax + DG_T - 1) / DG_T, (Nmax + DG_T - 1) / DG_T, nodes * M), 256, 0, s>>>(n, l, Qin, Qout, dw, skip);
        GG_CHECK_LAUNCH();
        if (dbg_stage) {
            if (dbg_nonfinite(dw.lam[l & 1], M, n, n, s)) return -20 - l;
        }
    }
    // eigenvalues of the root are in lam[0]; eigenvectors of T (rows) in A
    gg_count_launch(1);
    dc_unscale_kernel<<<dim3(4, M), 256, 0, s>>>(dw.lam[0], scale, n, D, skip);
    if (bt_side) gg_join(*bt_side, s, 1);
    if (stop_after == 2) return 0;

    // ---- stage 3 ----
    if (use_big) {
        // U (Delta matrices of the D&C stage) is free now: Y lives there
        double* Yb = dw.U;
        const int nt64 = (n + BB_T - 1) / BB_T;
        for (int P = npb - 1; P >= 0; --P) {
            const int len = n - (P * BB_NB + 1);
            gg_count_launch(1);
            bb_y_kernel<<<dim3(BB_NB / BB_T, nt64, M), 256, 0, s>>>(A, tw.Vh, n, P, Yb, skip);
            gg_count_launch(1);
            bb_upd_kernel<<<dim3((len + BB_T - 1) / BB_T, nt64, M), 256, 0, s>>>(A, Vp, Yb, n, P, skip);
        }
    } else if (npanels > 0 && which != 4) {
        gg_count_launch(1);
        bt_larft_kernel<<<dim3(npanels, M), 256, 0, s>>>(tw.Vh, tw.tau, n, Tm, npanels, skip);
        gg_count_launch(1);
        bt_apply_kernel<<<dim3((n + BT_R - 1) / BT_R, M), 256, 0, s>>>(A, tw.Vh, Tm, n, npanels, skip);
    }
    GG_CHECK_LAUNCH();
    return 0;
}
